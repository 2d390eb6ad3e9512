"""Top-C selection and scoring kernels at the count bounds of their loops and every width, against float64.

test_gpu_topc.py and test_gpu_topc_adapted.py hold the top-C kernels to the float64 definition on small shapes, where
no loop that carries state or strides across a grid runs past its first iteration.  This file takes those loops:

* ``topc_hist_kernel`` / ``topc_scatter_kernel`` (grid-stride over the (frame, slot) pairs) and ``topc_finalize_kernel``
  (grid-stride over (utterance, model)): grids capped at 4096 x 256 threads, crossed by T * C and n_utts * S.
* ``topc_scan_kernel``: one thread sums ceil(K / 1024) counts; K around 1024 and 2048.
* ``topc_product_kernel`` / ``topc_adapted_product_kernel``: the routed pairs of a component staged 64 at a time, with
  a tail batch; crafted selections route exactly n pairs to a component, through the C ABI.  Every mean-only width.
* ``topc_combine_kernel``: 64-frame groups walking ~300 000 utterances with runs of consecutive empty ones; entries of
  idx outside [0, K) (skipped) and a frame with no valid slot (-inf, as is its utterance).
* ``gmm_em_post_kernel<topc>`` with many images per CTA, ``em_topc_merge_kernel``'s grid-stride loop, and the selection
  on ragged segments (the plan kernel's padding and scan, dead rows), bit-equal to the selection on one segment.

The scores are held to ``score_given``, the float64 definition on a given selection: the scoring kernels on the
selection logits they are given (promoted to float64), and the frame values end to end on the float64 logits of the
GPU's selection.  Tolerances are those of test_gpu_topc.py.  Every GPU test prints its largest
errors (profiles/r3h_pytest_gpu_topc_counts.log).  ``test_count_lists_straddle_every_topc_bound`` parses the bounds out
of the CUDA sources and checks that the cases below sit on both sides of each.
"""
import ctypes as C
import functools
import re

import numpy as np
import pytest

from oracle import gmm as ogmm
from speech_signal_processing_b200 import synth
from test_gpu_gmm_counts import _int, _offsets, _source, _straddles
from test_gpu_topc import LLR_ATOL, SCORE_RTOL, check_selection, shared_set
from test_topc_adapted_host import score_top_c_adapted
from test_topc_host import case, score_top_c, top_components

FRAME_RTOL = 5e-5      # per-frame values, relative to max(1, |value|): the bound of test_gpu_topc.py's check_scores


# ------------------------------------------------------------------------------------------------ kernel counts
@functools.lru_cache(maxsize=None)
def topc_counts():
    """The loop bounds of the top-C kernels, parsed out of the CUDA sources (on first use, so that a pattern that stops
    matching fails the tests that need it, not the collection of this file)."""
    topc, common, em = (_source(n) for n in ("gmm_topc.cu", "common.cuh", "gmm_em_tc.cu"))
    nq = {name: sorted(int(v) for v in re.findall(r"SSP_TOPC_PRODUCT\((\d+)\)", body))
          for body, name in re.findall(r"switch \(DA / 4\) \{(.*?)default: SSP_REQUIRE\(false, \"(\w+):", topc, re.S)}
    assert set(nq) == {"ssp_gmm_score_topc", "ssp_gmm_score_topc_adapted"}, "the two product switches"
    for name, v in nq.items():
        assert v == list(range(1, len(v) + 1)), (name, v)
    return {
        "kThreads": _int(r"constexpr int kThreads = (\d+);", topc),
        "kBatch": _int(r"constexpr int kBatch = (\d+);", topc),
        "kCombineFrames": _int(r"constexpr int kCombineFrames = (\d+);", topc),
        "kTopcChunkFrames": _int(r"constexpr int64_t kTopcChunkFrames = (\d+);", common),
        "kTopcMaxC": _int(r"constexpr int kTopcMaxC = (\d+);", common),
        "kTopcMaxFeat": _int(r"constexpr int kTopcMaxFeat = (\d+);", common),
        "PAIR_GRID_CAP": _int(r"g_pairs = \(unsigned\)std::min<int64_t>\(\(pairs \+ 255\) / 256, (\d+)\);", topc),
        "HIST_THREADS": _int(r"topc_hist_kernel<<<g_pairs, (\d+),", topc),
        "SCATTER_THREADS": _int(r"topc_scatter_kernel<<<g_pairs, (\d+),", topc),
        "FINALIZE_GRID_CAP": _int(r"g = \(unsigned\)std::min<int64_t>\(\(n_utts \* S \+ 255\) / 256, (\d+)\);", topc),
        "FINALIZE_THREADS": _int(r"topc_finalize_kernel<<<g, (\d+),", topc),
        "SCAN_THREADS": _int(r"topc_scan_kernel<<<\(unsigned\)w\.n_chunks, (\d+),", topc),
        "SCAN_PER": _int(r"const int per = \(r\.K \+ \d+\) / (\d+);", topc),
        "SCAN_SHARED": _int(r"__shared__ int32_t part\[(\d+)\];", topc),
        "NQ_MEAN": nq["ssp_gmm_score_topc"][-1],
        "NQ_ADAPTED": nq["ssp_gmm_score_topc_adapted"][-1],
        "kTopcMergeThreads": _int(r"constexpr int kTopcMergeThreads = (\d+);", em),
        "MERGE_CTAS_PER_SM": _int(r"/ kTopcMergeThreads, cap = (\d+) \* \(int64_t\)g_num_sms;", em),
        "EM_BN": _int(r"constexpr int BN = (\d+);", em),
        "EM_IMG": _int(r"constexpr int IMG = (\d+);", em),
        "EM_BLK": _int(r"constexpr int BLK = (\d+);", em),
        "EM_NS_L": _int(r"constexpr int NS_L = (\d+);", em),
        "EM_PLAN_THREADS": _int(r"em_plan_kernel<<<1, (\d+),", em),
    }


# the values the cases of this file were written for: a change to one of them fails here until the cases follow
PINNED = {"kThreads": 128, "kBatch": 64, "kCombineFrames": 64, "kTopcChunkFrames": 4096, "kTopcMaxC": 64,
          "kTopcMaxFeat": 39, "PAIR_GRID_CAP": 4096, "HIST_THREADS": 256, "SCATTER_THREADS": 256,
          "FINALIZE_GRID_CAP": 4096, "FINALIZE_THREADS": 256, "SCAN_THREADS": 1024, "SCAN_PER": 1024,
          "SCAN_SHARED": 1024, "NQ_MEAN": 10, "NQ_ADAPTED": 20, "kTopcMergeThreads": 128, "MERGE_CTAS_PER_SM": 8,
          "EM_BN": 128, "EM_IMG": 128, "EM_BLK": 64, "EM_NS_L": 3, "EM_PLAN_THREADS": 1024}

# cases
CHUNK = PINNED["kTopcChunkFrames"]
ROUTED = (0, 1, 63, 64, 65, 127, 128, 129)   # pairs routed to one component in a chunk (crafted selections)
ROUTE_K, ROUTE_D, ROUTE_C = 64, 13, 5
GRID_UTTS = 300_000                          # utterances of 0 .. 3 frames (the grid-stride and combine case) ...
GRID_EMPTY_RUNS = (2, 3, 5, 17, 70)          # ... with runs of consecutive empty ones ...
GRID_LONG = (63, 64, 65, 63, 64, 65, CHUNK + 300)   # ... and a few long ones
GRID_K, GRID_D, GRID_C, GRID_S = 64, 13, 5, 4
SCAN_K = (1023, 1024, 1025, 2049)            # ceil(K / 1024) = 1, 1, 2, 3 counts per scan thread
WIDTH_K = (5, 129)
SEG_LENS = (0, 1, 63, 64, 65, 127, 128, 129) # selection on ragged segments ...
SEG_TINY = 2049                              # ... mixed into this many segments of 0 .. 3 frames
MANY_IMAGES = ((64, 300_000), (2048, 40_000))   # (K, T): many Fb images per CTA of the selection pass
SELECT_C = (1, 5, 64)
B200_SMS = 148                               # the guard's device; the GPU tests use the device's own count


def grid_lens():
    """GRID_UTTS utterances of 0 .. 3 frames: runs of GRID_EMPTY_RUNS consecutive empty utterances, among them three at
    the start of chunks and of 64-frame combine groups, the GRID_LONG utterances at seeded places, empty first and last."""
    rs = np.random.RandomState(17)
    lens = rs.randint(0, 4, size=GRID_UTTS)
    starts = rs.choice(np.arange(1, GRID_UTTS - 100), size=8 * len(GRID_EMPTY_RUNS), replace=False)
    for s, run in zip(starts, GRID_EMPTY_RUNS * 8):
        lens[s : s + run] = 0
    pos = rs.choice(np.arange(1, GRID_UTTS - 1), size=len(GRID_LONG), replace=False)
    lens[pos] = GRID_LONG
    lens[0] = lens[-1] = 0
    offs = _offsets(lens)
    live = lens > 0
    at_chunk = np.flatnonzero(live & (offs[:-1] % CHUNK == 0) & (offs[:-1] > 0))[:3]
    at_group = np.flatnonzero(live & (offs[:-1] % PINNED["kCombineFrames"] == 0) & (offs[:-1] % CHUNK != 0))[:3]
    return np.insert(lens, np.repeat(np.concatenate([at_chunk, at_group]), 4), 0)


def images_per_cta(k, t, sms):
    """Fb images (128 frames) each CTA of the selection pass takes for one segment of t frames: the grid is
    (SMs / tile pairs) x tile pairs."""
    B = PINNED
    pairs = (-(-k // B["EM_BN"]) + 1) // 2
    images = -(-(-(-t // B["EM_BLK"])) // 2)
    gx = min(max(1, sms // pairs), images)
    return -(-images // gx)


def merge_passes(t, n_segs, sms):
    """Grid-stride passes of em_topc_merge_kernel: its grid is sized from the workspace's padded rows and capped at
    MERGE_CTAS_PER_SM x SMs CTAs."""
    B = PINNED
    rows = ((t // B["EM_BLK"] + 2 * n_segs + 2) & ~1) * B["EM_BLK"]
    blocks = -(-rows // B["kTopcMergeThreads"])
    grid = min(blocks, B["MERGE_CTAS_PER_SM"] * sms)
    used = -(-(-(-t // B["EM_BLK"]) + 1) // 2) * 2 * B["EM_BLK"]    # the rows the merge walks (one segment)
    return -(-used // (grid * B["kTopcMergeThreads"]))


def test_count_lists_straddle_every_topc_bound():
    B = topc_counts()
    assert B == PINNED, "a top-C kernel bound changed: move the cases of this file with it"
    # product: a component's pairs in batches of kBatch, a tail batch or none, one and two batches; a whole chunk on one
    # component is kTopcChunkFrames / kBatch full batches
    b = B["kBatch"]
    assert {0, 1} <= set(ROUTED) and _straddles(ROUTED, b) and {2 * b - 1, 2 * b, 2 * b + 1} <= set(ROUTED)
    assert sum(ROUTED) <= B["kTopcChunkFrames"] and B["kTopcChunkFrames"] % b == 0 and B["kTopcChunkFrames"] // b > 2
    # hist / scatter and finalize stride past their capped grids; more than 100 chunks; the combine's groups
    lens = grid_lens()
    t, n_utts = int(lens.sum()), len(lens)
    assert t * GRID_C > 2 * B["PAIR_GRID_CAP"] * B["HIST_THREADS"] and B["HIST_THREADS"] == B["SCATTER_THREADS"]
    assert n_utts * GRID_S > B["FINALIZE_GRID_CAP"] * B["FINALIZE_THREADS"]
    assert -(-t // B["kTopcChunkFrames"]) > 100
    assert _straddles(GRID_LONG, B["kCombineFrames"]) and max(GRID_LONG) > B["kTopcChunkFrames"]
    empty = np.concatenate([[0], (lens == 0).astype(int), [0]])
    runs = np.flatnonzero(np.diff(empty) == -1) - np.flatnonzero(np.diff(empty) == 1)
    assert runs.max() > B["kCombineFrames"] and (runs >= 2).sum() > 10
    offs = _offsets(lens)
    for unit in (B["kTopcChunkFrames"], B["kCombineFrames"]):   # empty utterances where a chunk and a group start
        assert any(lens[u] == 0 and lens[u + 1] == 0 and offs[u] % unit == 0 and offs[u] > 0 for u in range(len(lens) - 1))
    # scan: 1, 2 and 3 counts per thread, K on both sides of the thread count
    n = B["SCAN_THREADS"]
    assert B["SCAN_PER"] == B["SCAN_SHARED"] == n and {n - 1, n, n + 1} <= set(SCAN_K)
    assert {-(-k // n) for k in SCAN_K} == {1, 2, 3}
    # every width of both product switches
    nq = {(d + 1 + 3) // 4 for d in range(1, B["kTopcMaxFeat"] + 1)}
    assert nq == set(range(1, B["NQ_MEAN"] + 1))
    assert {(2 * d + 1 + 3) // 4 for d in range(1, B["kTopcMaxFeat"] + 1)} == set(range(1, B["NQ_ADAPTED"] + 1))
    # selection: segments around the 64-frame blocks and 128-frame images, more segments than the plan's scan threads
    assert _straddles(SEG_LENS, B["EM_BLK"]) and _straddles(SEG_LENS, B["EM_IMG"]) and 0 in SEG_LENS
    assert SEG_TINY > 2 * B["EM_PLAN_THREADS"]
    # many images per CTA (the Fb ring of EM_NS_L stages and the 4 TMEM slots wrap), the merge strides (a 148-SM B200)
    assert all(images_per_cta(k, t, B200_SMS) > 4 * B["EM_NS_L"] for k, t in MANY_IMAGES)
    assert merge_passes(MANY_IMAGES[0][1], 1, B200_SMS) >= 2
    assert max(SELECT_C) == B["kTopcMaxC"] and min(SELECT_C) == 1


# ------------------------------------------------------------------------------------------------ float64 reference
def score_given(x, frame_offsets, idx, weights, means, variances, ref, logit=None, block=65536):
    """Top-C scores on a given selection ``idx`` (T, C), float64: for every model s and frame t

        l_s(t) = log sum_{valid j} exp(logit[t, j] + L_s,c(t) - L_r,c(t)),   c = idx[t, j],

    L = log w + log N of oracle/gmm.py for member s and the reference member ``ref`` of the stacks ``weights`` (S, K),
    ``means`` and ``variances`` (S, K, D).  ``logit`` (T, C) is the given selection logit, promoted to float64; None
    takes the float64 L_r,c(t).  Slots with idx outside [0, K) are skipped; a frame without a valid slot is -inf, and so
    is the score of its utterance.  Utterance score = mean over its frames, 0 for an empty one.  Returns (scores
    (n_utts, S), frame values (S, T))."""
    x = np.asarray(x, dtype=np.float64)
    idx = np.asarray(idx, dtype=np.int64)
    n_models, k = np.shape(weights)
    valid = (idx >= 0) & (idx < k)
    safe = np.where(valid, idx, 0)     # (take_along_axis would wrap -1 to the last component)
    frame = np.empty((n_models, len(x)))
    for t0 in range(0, len(x), block):
        sl = slice(t0, t0 + block)
        lr = np.take_along_axis(ogmm.weighted_log_prob(x[sl], weights[ref], means[ref], variances[ref]), safe[sl], axis=1)
        base = lr if logit is None else np.asarray(logit[sl], dtype=np.float64)
        for s in range(n_models):
            ls = np.take_along_axis(ogmm.weighted_log_prob(x[sl], weights[s], means[s], variances[s]), safe[sl], axis=1)
            v = np.where(valid[sl], base + (ls - lr), -np.inf)
            m = v.max(axis=1)
            m0 = np.where(np.isfinite(m), m, 0.0)
            with np.errstate(divide="ignore"):
                frame[s, sl] = m0 + np.log(np.exp(v - m0[:, None]).sum(axis=1))
    offs = np.asarray(frame_offsets, dtype=np.int64)
    lens = np.diff(offs)
    scores = np.zeros((len(lens), n_models))
    live = lens > 0
    if live.any():
        scores[live] = (np.add.reduceat(frame, offs[:-1][live], axis=1) / lens[live]).T
    return scores, frame


def test_reference_equals_the_definitions_on_valid_selections():
    x, offs, w, var, means = case(s=4, k=12, d=5, lens=(30, 0, 1, 17))
    s = len(means)
    W, V = np.broadcast_to(w, (s,) + w.shape), np.broadcast_to(var, (s,) + var.shape)
    sw = W * np.random.RandomState(3).uniform(0.5, 1.5, size=W.shape)
    sv = V * np.random.RandomState(4).uniform(0.6, 1.6, size=V.shape)
    sw[3], sv[3] = w, var
    for c in (1, 3, 12):
        idx, logit = top_components(x, w, means[3], var, c)
        want, want_frame = score_top_c(x, offs, w, var, means, 3, c, idx=idx)
        for lg in (None, logit):
            got, got_frame = score_given(x, offs, idx, W, means, V, 3, logit=lg, block=7)
            np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-12)
            np.testing.assert_allclose(got_frame, want_frame, rtol=1e-12, atol=1e-12)
        want, want_frame = score_top_c_adapted(x, offs, sw, means, sv, 3, c, idx=idx)
        got, got_frame = score_given(x, offs, idx, sw, means, sv, 3)
        np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(got_frame, want_frame, rtol=1e-12, atol=1e-12)


def test_reference_skips_invalid_slots_and_counts_duplicates():
    x, offs, w, var, means = case(s=3, k=12, d=5, lens=(10, 1, 0, 9))
    s = len(means)
    W, V = np.broadcast_to(w, (s,) + w.shape), np.broadcast_to(var, (s,) + var.shape)
    idx, logit = top_components(x, w, means[2], var, 3)
    two, two_frame = score_given(x, offs, idx[:, :2], W, means, V, 2, logit=logit[:, :2])
    cut = idx.copy()
    cut[:, 2] = np.where(np.arange(len(x)) % 2, -1, 12)       # the last slot skipped: the C = 2 values
    lg = logit.copy()
    lg[:, 2] = np.nan                                           # never read
    got, got_frame = score_given(x, offs, cut, W, means, V, 2, logit=lg)
    np.testing.assert_array_equal(got_frame, two_frame)
    np.testing.assert_array_equal(got, two)
    # a frame without a valid slot: -inf, and so is its utterance (the one-frame utterance 1); the others are unchanged
    cut[10] = [-1, 12, -7]
    got, got_frame = score_given(x, offs, cut, W, means, V, 2, logit=lg)
    assert (got_frame[:, 10] == -np.inf).all() and (got[1] == -np.inf).all()
    np.testing.assert_array_equal(got[[0, 2, 3]], two[[0, 2, 3]])
    # a component in two slots of a frame counts twice
    dup = idx.copy()
    dup[:, 1] = dup[:, 0]
    lgd = logit.copy()
    lgd[:, 1] = lgd[:, 0]
    _, got_frame = score_given(x, offs, dup, W, means, V, 2, logit=lgd)
    _, one = score_given(x, offs, idx[:, :1], W, means, V, 2, logit=logit[:, :1])
    _, third = score_given(x, offs, idx[:, 2:], W, means, V, 2, logit=logit[:, 2:])
    np.testing.assert_allclose(got_frame, np.logaddexp(one + np.log(2.0), third), rtol=1e-14)


# ------------------------------------------------------------------------------------------------ crafted routing
TARGETS = len(ROUTED)   # components 0 .. 7 get ROUTED[i] pairs in chunk 0 and ROUTED[-1 - i] in chunk 2
FULL = TARGETS          # component 8 is slot 0 of every frame of chunk 1: a full chunk of kBatch-sized batches


def crafted_routing(k, c, mu, var, seed):
    """A selection over three chunks and 517 frames of a fourth, built so that a chosen component receives exactly n
    pairs of a chunk.  Every frame has a home component from which its features are drawn, placed in one of its slots
    (so that slot dominates the frame's value); the other slots hold filler components (> FULL).  Target homes: n of
    ROUTED in chunk 0 and chunk 2, FULL in all of chunk 1.  Among the filler-home frames, 60 hold their home twice,
    300 have a slot outside [0, K) (-1 or K), and one (in chunk 2) has no valid slot.  Returns (x (T, D) float32,
    idx (T, C) int32, offsets, {"bad": that frame, "target_pairs": [(component, frames of its pairs in chunk 0)]})."""
    t_all = 3 * CHUNK + 517
    rs = np.random.RandomState(seed)
    fillers = np.arange(FULL + 1, k)
    home = rs.choice(fillers, size=t_all)
    for ch, counts in ((0, ROUTED), (2, ROUTED[::-1])):
        h = np.concatenate([np.full(n, i) for i, n in enumerate(counts)])
        home[ch * CHUNK + rs.choice(CHUNK, size=len(h), replace=False)] = h
    home[CHUNK : 2 * CHUNK] = FULL
    x = (mu[home] + np.sqrt(var[home]) * rs.standard_normal((t_all, mu.shape[1]))).astype(np.float32)
    idx = rs.choice(fillers, size=(t_all, c))
    slot = rs.randint(0, c, size=t_all)
    slot[CHUNK : 2 * CHUNK] = 0
    rows = np.arange(t_all)
    idx[rows, slot] = home
    free = rs.permutation(np.flatnonzero(home > FULL))
    dup, inv = free[:60], free[60:360]
    idx[dup, (slot[dup] + 1) % c] = home[dup]
    idx[inv, (slot[inv] + 1 + rs.randint(0, c - 1, size=len(inv))) % c] = np.where(rs.rand(len(inv)) < 0.5, -1, k)
    bad = int(free[360:][(free[360:] >= 2 * CHUNK) & (free[360:] < 3 * CHUNK)][0])
    idx[bad] = np.where(np.arange(c) % 2, k, -1)
    # the counts the cases are about
    valid = (idx >= 0) & (idx < k)
    def counts(ch):
        sl = slice(ch * CHUNK, (ch + 1) * CHUNK)
        return np.bincount(idx[sl][valid[sl]], minlength=k)
    assert tuple(counts(0)[:TARGETS]) == ROUTED and tuple(counts(2)[:TARGETS]) == ROUTED[::-1]
    assert counts(1)[FULL] == CHUNK and counts(0)[FULL] == counts(2)[FULL] == 0
    cuts = rs.choice(np.arange(1, t_all), size=60, replace=False)
    cuts = np.concatenate([[0, t_all, bad, bad + 1, CHUNK, 2 * CHUNK, 3 * CHUNK], cuts, cuts[:6]])   # six empties
    offs = np.sort(cuts).astype(np.int64)
    targets = [(i, np.flatnonzero(home[:CHUNK] == i)) for i in range(TARGETS)]
    return x, idx.astype(np.int32), offs, {"bad": bad, "target_pairs": targets}


def routing_case(adapted, seed=5):
    """(x, idx, offsets, info, (w, mu, var) stacks (S = 4, the UBM last), float32 selection logits of the UBM with NaN in
    the skipped slots)."""
    k, d, c = ROUTE_K, ROUTE_D, ROUTE_C
    w, var, means = shared_set(4, k, d, seed=seed)
    W, V = np.tile(w, (4, 1)), np.tile(var, (4, 1, 1))
    if adapted:
        rs = np.random.RandomState(seed + 1)
        W[:3] *= rs.uniform(0.5, 1.5, size=(3, k))
        W[:3] /= W[:3].sum(axis=1, keepdims=True)
        V[:3] *= rs.uniform(0.6, 1.6, size=(3, k, d))
    x, idx, offs, info = crafted_routing(k, c, means[-1], var, seed)
    valid = (idx >= 0) & (idx < k)
    lr = ogmm.weighted_log_prob(x, W[-1], means[-1], V[-1])
    logit = np.where(valid, np.take_along_axis(lr, np.where(valid, idx, 0), axis=1), np.nan).astype(np.float32)
    return x, idx, offs, info, (W, means, V), logit


def test_the_reference_sees_a_dropped_tail_batch_and_a_shifted_chunk():
    """What the crafted-routing test would see of two slips of a product kernel, on the float64 side: the tail batch of
    every component whose count in chunk 0 is not a multiple of kBatch left out, and chunk 2's frames read one frame
    late.  Both move the affected frames and utterances far outside the tolerances."""
    x, idx, offs, info, (W, M, V), logit = routing_case(adapted=False)
    want, want_frame = score_given(x, offs, idx, W, M, V, 3, logit=logit)
    b = PINNED["kBatch"]
    drop = idx.copy()
    for comp, frames in info["target_pairs"]:
        tail = frames[len(frames) - len(frames) % b :]
        drop[tail] = np.where(drop[tail] == comp, -1, drop[tail])
    got, got_frame = score_given(x, offs, drop, W, M, V, 3, logit=logit)
    with np.errstate(invalid="ignore"):   # the frame without a valid slot: -inf on both sides
        frame_err = np.abs(got_frame - want_frame) / np.maximum(1.0, np.abs(want_frame))
        rel = np.abs(got - want) / np.maximum(1.0, np.abs(want))
    # the check takes the largest error: the tail of every component is seen on its own
    for comp, frames in info["target_pairs"]:
        tail = frames[len(frames) - len(frames) % b :]
        if len(tail):
            utts = np.searchsorted(offs, tail, side="right") - 1
            fe, ue = np.nanmax(frame_err[:, tail]), np.nanmax(rel[utts])
            print(f"tail of {len(tail)} of component {comp}'s {len(frames)} pairs dropped: frame values {fe:.2e} rel, "
                  f"scores {ue:.2e} rel")
            assert fe > 100 * FRAME_RTOL and ue > 10 * SCORE_RTOL
    late = x.copy()
    late[2 * CHUNK : 3 * CHUNK] = x[2 * CHUNK + 1 : 3 * CHUNK + 1]
    _, got_frame = score_given(late, offs, idx, W, M, V, 3, logit=logit)
    spk = (slice(0, 3), slice(2 * CHUNK, 3 * CHUNK))   # the speakers (the reference member's values are the logits)
    ok = np.isfinite(want_frame[spk])
    frame_err = np.abs(got_frame[spk][ok] - want_frame[spk][ok]) / np.maximum(1.0, np.abs(want_frame[spk][ok]))
    print(f"chunk 2 one frame late: {np.mean(frame_err > 100 * FRAME_RTOL):.3f} of the speakers' frame values there "
          "outside 100 x the bound")
    assert np.mean(frame_err > 100 * FRAME_RTOL) > 0.9


# ------------------------------------------------------------------------------------------------ GPU helpers
def _torch():
    from speech_signal_processing_b200 import _lib

    return _lib.require_cuda()


def _dev(a, dtype=None):
    return _torch().as_tensor(np.ascontiguousarray(a), dtype=dtype, device="cuda")


def check(case_name, got, lse, want, want_frame, ref, offs, frame64=None):
    """Scores (relative), LLRs against the reference member (absolute) and frame values (relative) against float64 on
    the same selection logits; -inf where the reference is -inf, and 0 for empty utterances.  ``frame64``: the frame
    values on float64 selection logits, held to the frame bound (end to end: the FP32-grade logits of the selection
    included).  Returns the largest errors."""
    inf_f, inf_u = np.isinf(want_frame), np.isinf(want)
    assert (want_frame[inf_f] == -np.inf).all() and (want[inf_u] == -np.inf).all()
    assert (lse[inf_f] == -np.inf).all() and (got[inf_u] == -np.inf).all(), case_name
    assert np.isfinite(lse[~inf_f]).all() and np.isfinite(got[~inf_u]).all(), case_name
    u = ~inf_u.any(axis=1)
    rel = float((np.abs(got[u] - want[u]) / np.maximum(1.0, np.abs(want[u]))).max())
    llr = float(np.abs((got[u] - got[u, ref : ref + 1]) - (want[u] - want[u, ref : ref + 1])).max())
    fr = float((np.abs(lse[~inf_f] - want_frame[~inf_f]) / np.maximum(1.0, np.abs(want_frame[~inf_f]))).max()) \
        if (~inf_f).any() else 0.0
    extra = f", {int(inf_u.any(axis=1).sum())} utterances and {int(inf_f.any(axis=0).sum())} frames -inf" if inf_f.any() else ""
    if frame64 is not None and (~inf_f).any():
        assert (np.isinf(frame64) == inf_f).all()
        fr64 = float((np.abs(lse[~inf_f] - frame64[~inf_f]) / np.maximum(1.0, np.abs(frame64[~inf_f]))).max())
    else:
        fr64 = 0.0
    if frame64 is not None:
        extra += f"; end to end (float64 selection logits) frame values {fr64:.2e} rel"
    print(f"{case_name}: scores {rel:.2e} rel, LLR {llr:.2e} abs, frame values {fr:.2e} rel{extra}")
    assert rel <= SCORE_RTOL, case_name
    assert llr <= LLR_ATOL, case_name
    assert fr <= FRAME_RTOL, case_name
    assert fr64 <= FRAME_RTOL, case_name
    assert (got[np.diff(offs) == 0] == 0.0).all(), case_name
    return rel, llr, fr


def check_reference_lse(case_name, lse_ref, logit, idx, k):
    """The reference member's row of the table is zeros, so its frame values are m + logf(sum __expf(logit - m)) over
    the valid slots of the given FP32 logits: within the __expf error (~2^-22 per term), the FP32 sum's rounding (2^-24
    per add) and logf's, plus half an ulp of the result, of the float64 log-sum-exp.  -inf for a frame without a valid
    slot."""
    valid = (idx >= 0) & (idx < k)
    v = np.where(valid, logit.astype(np.float64), -np.inf)
    m = v.max(axis=1)
    m0 = np.where(np.isfinite(m), m, 0.0)
    with np.errstate(divide="ignore"):
        want = m0 + np.log(np.exp(v - m0[:, None]).sum(axis=1))
    live = np.isfinite(want)
    assert (lse_ref[~live] == -np.inf).all(), case_name
    err = np.abs(lse_ref[live].astype(np.float64) - want[live])
    bound = 2.0 ** -24 * np.abs(want[live]) + (idx.shape[1] + 8) * 2.0 ** -23
    print(f"{case_name}: reference member's frame values vs the log-sum-exp of the given logits: "
          f"{float((err / bound).max()):.2f} of the FP32 bound")
    assert (err <= bound).all(), case_name


def stacks(ms):
    """(weights (S, K), means, variances (S, K, D), reference member) of a SharedModelSet or a with_ubm ModelSet."""
    import speech_signal_processing_b200 as ssp

    if isinstance(ms, ssp.SharedModelSet):
        w, var, mu = (t.cpu().numpy() for t in ms._params)
        s = mu.shape[0]
        return np.broadcast_to(w, (s,) + w.shape), mu, np.broadcast_to(var, (s,) + var.shape), ms.ref_model
    w, mu, var = (t.cpu().numpy() for t in ms._params)
    return w, mu, var, ms.ubm_index


def score_public(case_name, ms, x, offs, c, feats=None):
    """score_top_c of a SharedModelSet or with_ubm ModelSet against score_given on the GPU's own selection: scores,
    LLRs and frame values on its logits, and the frame values on float64 logits (test_gpu_topc.py's check).  The
    utterance bound SCORE_RTOL is for the scoring kernels: end to end, the score of a one-frame utterance is a frame
    value, with the selection logit's FP32-grade error in it, which only the frame bound covers.  Returns (scores,
    frame values, selection idx, selection logits)."""
    feats = _dev(x) if feats is None else feats
    got, lse = ms.score_top_c(feats, offs, c=c, want_frame_lse=True)
    idx, logit = ms._topc[0].top_components(feats, np.array([0, len(x)]), c)
    idx, logit = idx.cpu().numpy(), logit.cpu().numpy()
    w, mu, var, ref = stacks(ms)
    want, want_frame = score_given(x, offs, idx, w, mu, var, ref, logit=logit)
    _, frame64 = score_given(x, offs, idx, w, mu, var, ref)
    got, lse = got.cpu().numpy(), lse.cpu().numpy()
    check(case_name, got, lse, want, want_frame, ref, offs, frame64=frame64)
    return got, lse, idx, logit


def synthetic_adapted(n_spk, k, d, seed):
    from test_gpu_topc_adapted import synthetic_set

    return synthetic_set(n_spk, k, d, seed)


# ------------------------------------------------------------------------------------------------ crafted routing (C ABI)
@pytest.mark.gpu
@pytest.mark.parametrize("adapted", [False, True], ids=["mean-only", "adapted"])
def test_crafted_routing_through_the_c_abi(adapted):
    """ssp_gmm_pack_topc[_adapted] and ssp_gmm_score_topc[_adapted] on a crafted selection: a component receives 0, 1,
    63, 64, 65, 127, 128 and 129 pairs of chunk 0 and of chunk 2 (the product kernels' 64-pair batches and their tail),
    one component every frame of chunk 1 (64 full batches); skipped slots (-1, K, their logits NaN), duplicates, and a
    frame with no valid slot.  The workspace starts as NaN bytes.  Against score_given on the given float32 logits."""
    from speech_signal_processing_b200 import _lib

    torch = _torch()
    lib = _lib.load()
    x, idx, offs, info, (W, M, V), logit = routing_case(adapted)
    s, k, d = M.shape
    c = idx.shape[1]
    dims = _lib.GmmDims(s, k, d)
    ref = s - 1
    if adapted:
        nbytes = int(lib.ssp_gmm_topc_adapted_pack_bytes(C.byref(dims)))
        assert nbytes == (k * s * ((2 * d + 1 + 3) // 4 * 4) + k * ((d + 3) // 4 * 4)) * 4
        pack = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
        pw, pm, pv = _dev(W, torch.float64), _dev(M, torch.float64), _dev(V, torch.float64)
        _lib.check(lib.ssp_gmm_pack_topc_adapted(pw.data_ptr(), pm.data_ptr(), pv.data_ptr(), C.byref(dims), ref,
                                                 pack.data_ptr(), _lib.stream_ptr()), "ssp_gmm_pack_topc_adapted")
        score, name, product = lib.ssp_gmm_score_topc_adapted, "ssp_gmm_score_topc_adapted", "topc_adapted_product_kernel"
    else:
        nbytes = int(lib.ssp_gmm_topc_pack_bytes(C.byref(dims)))
        assert nbytes == k * s * ((d + 1 + 3) // 4 * 4) * 4
        pack = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
        pv, pm = _dev(V[0], torch.float64), _dev(M, torch.float64)
        _lib.check(lib.ssp_gmm_pack_topc(pv.data_ptr(), pm.data_ptr(), C.byref(dims), ref, pack.data_ptr(),
                                         _lib.stream_ptr()), "ssp_gmm_pack_topc")
        score, name, product = lib.ssp_gmm_score_topc, "ssp_gmm_score_topc", "topc_product_kernel"
    t, n_utts = len(x), len(offs) - 1
    ws_bytes = int(lib.ssp_gmm_score_topc_workspace_bytes(C.byref(dims), c, t))
    ws = torch.full((ws_bytes,), 255, dtype=torch.uint8, device="cuda")
    feats, d_off, d_idx, d_logit = _dev(x), _dev(offs), _dev(idx), _dev(logit)
    scores = torch.empty((n_utts, s), dtype=torch.float64, device="cuda")
    lse = torch.empty((s, t), dtype=torch.float32, device="cuda")
    lib.ssp_reset_launch_count()
    _lib.check(score(feats.data_ptr(), d_off.data_ptr(), n_utts, t, d_idx.data_ptr(), d_logit.data_ptr(), c,
                     pack.data_ptr(), C.byref(dims), scores.data_ptr(), lse.data_ptr(), ws.data_ptr(), ws_bytes,
                     _lib.stream_ptr()), name)
    log = _lib.launch_log()
    n_chunks = -(-t // CHUNK)
    assert log[product] == n_chunks and log["topc_combine_kernel"] == n_chunks, log
    want, want_frame = score_given(x, offs, idx, W, M, V, ref, logit=logit)
    got, got_lse = scores.cpu().numpy(), lse.cpu().numpy()
    bad = info["bad"]
    assert (want_frame[:, bad] == -np.inf).all() and np.isinf(want).any()
    check(f"crafted routing {name}", got, got_lse, want, want_frame, ref, offs)
    check_reference_lse(f"crafted routing {name}", got_lse[ref], logit, idx, k)


# ------------------------------------------------------------------------------------------------ grid-stride loops
@pytest.mark.gpu
@pytest.mark.parametrize("form", ["shared", "adapted"])
def test_grid_strides_and_many_tiny_utterances(form):
    """~300 000 utterances of 0 .. 3 frames with runs of empty ones, some of 63 / 64 / 65 frames and one longer than a
    chunk: T * C > 2 x 4096 x 256 (hist and scatter stride at least twice), n_utts * S > 4096 x 256 (finalize strides),
    over 100 chunks, and the combine's groups walk several consecutive empty utterances."""
    import speech_signal_processing_b200 as ssp

    k, d, c, s = GRID_K, GRID_D, GRID_C, GRID_S
    lens = grid_lens()
    offs = _offsets(lens)
    if form == "shared":
        w, var, means = shared_set(s, k, d, seed=31)
        ms = ssp.SharedModelSet(w, var, means, ref_model=-1)
        x = synth.sample_gmm(w, means[-1], var, int(offs[-1]), seed=32)
    else:
        ms, (w, mu, var) = synthetic_adapted(s - 1, k, d, seed=31)
        x = synth.sample_gmm(w, mu, var, int(offs[-1]), seed=32)
    assert ms.n_models == s
    score_public(f"{form}: {len(lens)} utterances, {len(x)} frames, {-(-len(x) // CHUNK)} chunks", ms, x, offs, c)


# ------------------------------------------------------------------------------------------------ scan
@pytest.mark.gpu
@pytest.mark.parametrize("form", ["shared", "adapted"])
@pytest.mark.parametrize("k", SCAN_K)
def test_scan_at_one_two_and_three_counts_per_thread(k, form):
    """topc_scan_kernel gives each of its 1024 threads ceil(K / 1024) counts of a chunk to sum: K = 1023, 1024, 1025
    and 2049, T just over two chunks."""
    import speech_signal_processing_b200 as ssp

    d, c, s = 13, 5, 4
    lens = [0, 1, 300, CHUNK, 65, 0, CHUNK - 329]
    offs = _offsets(lens)
    if form == "shared":
        w, var, means = shared_set(s, k, d, seed=k)
        ms = ssp.SharedModelSet(w, var, means, ref_model=-1)
        x = synth.sample_gmm(w, means[-1], var, int(offs[-1]), seed=k + 1)
    else:
        ms, (w, mu, var) = synthetic_adapted(s - 1, k, d, seed=k)
        x = synth.sample_gmm(w, mu, var, int(offs[-1]), seed=k + 1)
    score_public(f"{form} K={k} ({-(-k // 1024)} counts per scan thread) T={len(x)}", ms, x, offs, c)


# ------------------------------------------------------------------------------------------------ widths
@pytest.mark.gpu
@pytest.mark.parametrize("k", WIDTH_K)
@pytest.mark.parametrize("d", list(range(1, PINNED["kTopcMaxFeat"] + 1)))
def test_every_mean_only_width(d, k):
    """topc_product_kernel<NQ> for NQ = 1 .. 10 (D = 1 .. 39), as test_gpu_topc_adapted.py does for the adapted form."""
    import speech_signal_processing_b200 as ssp

    w, var, means = shared_set(5, k, d, seed=d)
    sms = ssp.SharedModelSet(w, var, means, ref_model=-1)
    offs = _offsets([150, 0, 1, 210])
    x = synth.sample_gmm(w, means[-1], var, int(offs[-1]), seed=d + k)
    feats = _dev(x)
    for c in (1, min(k, 64)):
        score_public(f"D={d} (NQ={(d + 1 + 3) // 4}) K={k} C={c}", sms, x, offs, c, feats=feats)


# ------------------------------------------------------------------------------------------------ reference member
@pytest.mark.gpu
@pytest.mark.parametrize("ref", [0, 2])
def test_reference_member_and_exact_zeros(ref):
    """SharedModelSet(ref_model=ref) with a speaker whose means are the reference's (twin, in the same 32-byte sector of
    the score rows, so its double atomics meet the reference's in the same order).  The twin's frame values and scores
    equal the reference's bit for bit, its LLR is exactly 0.0, and the reference's frame values are the log-sum-exp of
    the selection logits to FP32 rounding (check_reference_lse)."""
    import speech_signal_processing_b200 as ssp

    k, d, c, s = 64, 13, 5, 4
    w, mu, var = synth.synth_ubm(k, d, seed=40 + ref, spread=1.0)
    means = synth.synth_speaker_means(mu, s, seed=41 + ref, shift=0.35)
    twin = ref + 1
    means[ref], means[twin] = mu, mu.copy()
    sms = ssp.SharedModelSet(w, var, means, ref_model=ref)
    assert sms.ref_model == ref
    offs = _offsets([300, 0, 1, 64, 65, CHUNK + 11, 0, 5])
    x = synth.sample_gmm(w, mu, var, int(offs[-1]), seed=42)
    got, lse, idx, logit = score_public(f"ref_model={ref}", sms, x, offs, c)
    assert (got[:, twin] - got[:, ref] == 0.0).all()
    np.testing.assert_array_equal(lse[twin], lse[ref])
    check_reference_lse(f"ref_model={ref}", lse[ref], logit, idx, k)
    others = [m for m in range(s) if m not in (ref, twin)]
    assert (np.abs(got[:, others] - got[:, [ref]])[np.diff(offs) > 0] > 0).all()


# ------------------------------------------------------------------------------------------------ selection
def _check_selection_blocks(case_name, idx, logit, x, w, mu, var):
    """check_selection over frame blocks of at most 2^24 float64 logits."""
    block = max(1, 2 ** 24 // len(w))
    for t0 in range(0, len(x), block):
        sl = slice(t0, t0 + block)
        check_selection(f"{case_name} frames {t0}..{min(t0 + block, len(x))}", idx[sl], logit[sl], x[sl], w, mu, var)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [64, 129])
def test_selection_on_ragged_segments(k):
    """ModelSet.top_components on segments of 0, 1, 63, 64, 65, 127, 128 and 129 frames among 2049 segments of 0 .. 3
    frames: the plan kernel's 1024-thread scan, segments padded to 64-frame blocks, dead rows skipped by the merge.  The
    result is bit-equal to the selection of the same frames as one segment (a row's logits do not depend on where the
    row sits in an image), and against float64 per frame."""
    import speech_signal_processing_b200 as ssp

    d = 13
    w, mu, var = synth.synth_ubm(k, d, seed=50 + k, spread=1.0)
    rs = np.random.RandomState(k)
    lens = rs.randint(0, 4, size=SEG_TINY)
    lens[rs.choice(np.arange(1, SEG_TINY - 1), size=len(SEG_LENS), replace=False)] = SEG_LENS
    offs = _offsets(lens)
    x = synth.sample_gmm(w, mu, var, int(offs[-1]), seed=51)
    ms = ssp.ModelSet(w, mu, var)
    feats = _dev(x)
    ws_seg, ws_one = ssp.mixture.StatsWorkspace(ms.device), ssp.mixture.StatsWorkspace(ms.device)
    for n, c in enumerate((1, 5)):
        idx, logit = (a.cpu().numpy() for a in ms.top_components(feats, offs, c, workspace=ws_seg, reuse_images=n > 0))
        one_idx, one_logit = (a.cpu().numpy() for a in ms.top_components(feats, [0, len(x)], c, workspace=ws_one,
                                                                           reuse_images=n > 0))
        np.testing.assert_array_equal(idx, one_idx)
        np.testing.assert_array_equal(logit, one_logit)
        check_selection(f"K={k} C={c} {len(lens)} segments, {len(x)} frames (bit-equal to one segment)", idx, logit, x,
                        w, mu, var)


@pytest.mark.gpu
@pytest.mark.parametrize("k,t", MANY_IMAGES)
def test_selection_with_many_images_per_cta(k, t):
    """gmm_em_post_kernel<topc> with ~16-18 Fb images per CTA (the Fb ring of 3 stages and the 4 TMEM slots wrap several
    times) and, at K = 64, em_topc_merge_kernel striding its capped grid; C = 1, 5 and 64 on the same images."""
    import speech_signal_processing_b200 as ssp

    torch = _torch()
    sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    per_cta = images_per_cta(k, t, sms)
    passes = merge_passes(t, 1, sms)
    assert per_cta > 4 * PINNED["EM_NS_L"]
    assert k > 64 or passes >= 2
    d = 13
    w, mu, var = synth.synth_ubm(k, d, seed=60 + k, spread=1.0)
    x = synth.sample_gmm(w, mu, var, t, seed=61)
    ms = ssp.ModelSet(w, mu, var)
    feats = _dev(x)
    ws = ssp.mixture.StatsWorkspace(ms.device)
    for n, c in enumerate(SELECT_C):
        idx, logit = (a.cpu().numpy() for a in ms.top_components(feats, [0, t], c, workspace=ws, reuse_images=n > 0))
        _check_selection_blocks(f"K={k} T={t} C={c} ({per_cta} images per CTA, {passes} merge passes)", idx, logit, x,
                                w, mu, var)
