"""Top-C fast scoring of speakers MAP-adapted in weights, means and variances against exact scoring at the headline shapes
on one GPU, one JSON line.

    python benchmarks/topc_adapted_bench.py [--seed 0] [--reps 5] [--warmup 1] [--device 0] [--utts 10000] [--check-utts 8]

Workload (config 4 shapes, generated on the device from the seed): a K = 1024, D = 39 UBM and 1 000 speakers enrolled by
``map_enrol(ubm, ..., adapt=("means", "weights", "variances"))`` at relevance 16 from 3 000 synthetic frames each, so
the set is a ``ModelSet`` of the speakers plus the UBM as member 1 000 (``ubm_index``).  Each speaker's frames come from
the UBM with shifted means and scaled variances, and --utts test utterances of 298 frames (2.98 M frames at the default)
are drawn the same way.  In one process, alternating call by call: exact ``ModelSet.score`` ("auto": one TF32 pass of the
general tensor kernel at K = 1024) and ``ModelSet.score_top_c`` at C = 1, 5 and 16, each timed with CUDA events over
--reps calls after --warmup (min / median / max), and the selection (``top_components`` of the UBM) on its own.
Reported as information, not as a criterion: how many decisions (argmax of the LLR against the UBM) agree between top-C
and exact scoring and the largest |LLR difference|.  Check: a float64 restatement of the adapted top-C score
(``reference_top_c_adapted``, held equal to the float64 definition in tests/test_topc_adapted_host.py) on --check-utts
seeded utterances, on the GPU's own selection.  Card name, power limit and maximum SM clock are read in the same run.
Writes nothing to the tree.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from benchmarks.topc_bench import C_VALUES, D, K, LLR_ATOL, N_SPK, UTT_FRAMES, gpu_info, stats  # noqa: E402

ENROL_FRAMES = 3000
RELEVANCE = 16.0


def reference_top_c_adapted(x, frame_offsets, weights, means, variances, idx):
    """float64 top-C scores (n_utts, S) of frames ``x`` (T, D) on the selection ``idx`` (T, C) for models with their own
    ``weights`` (S, K), ``means`` and ``variances`` (S, K, D): the mean over an utterance's frames of
    log sum_{c in idx[t]} w_s,c N(x_t; means[s, c], variances[s, c]); 0 for an empty utterance."""
    x = np.asarray(x, dtype=np.float64)
    w, mu, var = (np.asarray(a, dtype=np.float64) for a in (weights, means, variances))
    idx = np.asarray(idx, dtype=np.int64)
    xs = x[:, None, :]                                     # (T, 1, D)
    frame = np.empty((mu.shape[0], x.shape[0]))
    for s in range(mu.shape[0]):
        v = var[s][idx]                                    # (T, C, D)
        lp = np.log(w[s][idx]) - 0.5 * (x.shape[1] * np.log(2 * np.pi) + np.log(v).sum(axis=2)
                                        + (((xs - mu[s][idx]) ** 2) / v).sum(axis=2))
        m = lp.max(axis=1)
        frame[s] = m + np.log(np.exp(lp - m[:, None]).sum(axis=1))
    offs = np.asarray(frame_offsets, dtype=np.int64)
    out = np.zeros((len(offs) - 1, mu.shape[0]))
    for u in range(len(offs) - 1):
        if offs[u + 1] > offs[u]:
            out[u] = frame[:, offs[u] : offs[u + 1]].mean(axis=1)
    return out


def speaker_frames(torch, gen, dev, w, means, scale, spk, n_per):
    """``n_per`` frames of each speaker in ``spk`` (int64 device tensor): a component drawn from the UBM weights, the
    speaker's means and the UBM variances times the speaker's scale."""
    d_w, d_means, d_scale = (torch.as_tensor(a, device=dev) for a in (w, means, scale))
    spk = spk.repeat_interleave(n_per)
    comp = torch.multinomial(d_w, spk.numel(), replacement=True, generator=gen)
    sd = torch.sqrt(d_scale[spk, comp]).to(torch.float32)
    noise = torch.randn((spk.numel(), means.shape[2]), generator=gen, device=dev, dtype=torch.float32)
    return (d_means[spk, comp].to(torch.float32) + sd * noise).contiguous()


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--utts", type=int, default=10000)
    ap.add_argument("--check-utts", type=int, default=8)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("topc_adapted_bench.py measures the GPU kernels: no CUDA device found")
    import speech_signal_processing_b200 as ssp
    from speech_signal_processing_b200 import synth

    dev = torch.device("cuda", args.device)
    torch.cuda.set_device(dev)
    gpu = gpu_info(args.device)

    # ---- UBM, enrolment (weights, means and variances at relevance 16) and test frames
    w, mu, var = synth.synth_ubm(K, D, seed=args.seed)
    ubm = ssp.GaussianMixture.from_params(w, mu, var)
    true_means = synth.synth_speaker_means(mu, N_SPK, seed=args.seed + 1, shift=0.25)
    rs = np.random.RandomState(args.seed + 3)
    true_var = var[None] * rs.uniform(0.6, 1.5, size=(N_SPK, 1, D))
    gen = torch.Generator(device=dev)
    gen.manual_seed(args.seed)
    enrol = speaker_frames(torch, gen, dev, w, true_means, true_var, torch.arange(N_SPK, device=dev), ENROL_FRAMES)
    ms = ssp.map_enrol(ubm, (enrol, np.arange(N_SPK + 1, dtype=np.int64) * ENROL_FRAMES), relevance=RELEVANCE,
                       adapt=("means", "weights", "variances"), device=dev)
    del enrol
    T = args.utts * UTT_FRAMES
    spk = torch.randint(0, N_SPK, (args.utts,), generator=gen, device=dev)
    feats = speaker_frames(torch, gen, dev, w, true_means, true_var, spk, UTT_FRAMES)
    offs = np.arange(args.utts + 1, dtype=np.int64) * UTT_FRAMES

    # ---- timings, alternating the scorers call by call
    arms = {"exact": lambda: ms.score(feats, offs)}
    for c in C_VALUES:
        arms[f"top{c}"] = (lambda c=c: ms.score_top_c(feats, offs, c=c))
    ms.score_top_c(feats, offs, c=C_VALUES[0])            # builds the UBM set and the (a, b, k) table
    ref = ms._topc[0]
    whole = [0, T]
    arms["select5"] = lambda: ref.top_components(feats, whole, 5)
    times = {name: [] for name in arms}
    outs = {}
    for _ in range(args.warmup):
        for name, fn in arms.items():
            outs[name] = fn()
    torch.cuda.synchronize()
    for _ in range(args.reps):
        for name, fn in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            outs[name] = fn()
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1))

    # ---- agreement with exact scoring (information)
    u = ms.ubm_index

    def llr(scores):
        s = scores.cpu().numpy()
        return s[:, :u] - s[:, u : u + 1]

    exact = llr(outs["exact"][0])
    agree = {}
    for c in C_VALUES:
        got = llr(outs[f"top{c}"][0])
        agree[f"top{c}"] = {"decisions_equal": int((got.argmax(axis=1) == exact.argmax(axis=1)).sum()),
                            "utterances": int(args.utts), "max_abs_llr_diff": float(np.abs(got - exact).max())}

    # ---- float64 check of a seeded sample, on the GPU's own selection
    sw, smu, svar = (t.cpu().numpy() for t in ms._params)
    pick = np.sort(rs.choice(args.utts, size=min(args.check_utts, args.utts), replace=False))
    rows = np.concatenate([np.arange(p * UTT_FRAMES, (p + 1) * UTT_FRAMES) for p in pick])
    d_rows = torch.as_tensor(rows, device=dev)
    x = feats[d_rows].cpu().numpy()
    sub_offs = np.arange(len(pick) + 1, dtype=np.int64) * UTT_FRAMES
    check = {"utterances": int(len(pick))}
    for c in C_VALUES:
        idx, _ = ref.top_components(feats, whole, c)
        want = reference_top_c_adapted(x, sub_offs, sw, smu, svar, idx[d_rows].cpu().numpy())
        got = outs[f"top{c}"][0].cpu().numpy()[pick]
        check[f"top{c}"] = {"max_rel_score_err": float((np.abs(got - want) / np.maximum(1.0, np.abs(want))).max()),
                            "max_abs_llr_err": float(np.abs((got[:, :u] - got[:, u:]) - (want[:, :u] - want[:, u:])).max())}
    res = {
        "bench": "topc_adapted",
        "gpu": gpu,
        "shape": {"utterances": args.utts, "frames": T, "K": K, "D": D, "models": N_SPK + 1,
                  "enrolment": {"frames_per_speaker": ENROL_FRAMES, "relevance": RELEVANCE,
                                "adapt": ["means", "weights", "variances"]}},
        "ms": {name: stats(t) for name, t in times.items()},
        "speedup_vs_exact": {f"top{c}": float(np.median(times["exact"]) / np.median(times[f"top{c}"])) for c in C_VALUES},
        "agreement_with_exact": agree,
        "check_float64": check,
    }
    res["ok"] = all(check[f"top{c}"]["max_abs_llr_err"] <= LLR_ATOL for c in C_VALUES)
    print(json.dumps(res))
    return 0 if res["ok"] else 1


if __name__ == "__main__":
    sys.exit(main())
