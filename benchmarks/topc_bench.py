"""Top-C fast scoring against exact shared-variance scoring at the headline shapes on one GPU, one JSON line.

    python benchmarks/topc_bench.py [--seed 0] [--reps 5] [--warmup 1] [--device 0] [--utts 10000] [--check-utts 8]

Workload (config 4 shapes, generated on the device from the seed): a K = 1024, D = 39 UBM, 1 000 speakers whose means are
the UBM's shifted per component (what mean-only MAP enrolment yields) plus the UBM as member 1 000 and reference, and
--utts utterances of 298 frames (2.98 M frames at the default) drawn from the speakers.  In one process, alternating
call by call: exact ``SharedModelSet.score`` and ``score_top_c`` at C = 1, 5 and 16, each timed with CUDA events over
--reps calls after --warmup (min / median / max), and the selection (``ModelSet.top_components`` of the UBM) on its own.
Reported as information, not as a criterion: how many decisions (argmax of the LLR against the UBM) agree between top-C
and exact scoring and the largest |LLR difference|; the synthetic UBM is flat (about 45 components carry a frame), so
top-C moves further from exact than it does on speech.  Check: a float64 restatement of the top-C score
(``reference_top_c``, held equal to the float64 definition in tests/test_topc_host.py) on --check-utts seeded utterances, on the
GPU's own selection.  Card name, power limit and maximum SM clock are read in the same run.  Writes nothing to the tree.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

K, D, N_SPK, UTT_FRAMES = 1024, 39, 1000, 298
C_VALUES = (1, 5, 16)
LLR_ATOL = 1e-3


def reference_top_c(x, frame_offsets, weights, variances, means, idx):
    """float64 top-C scores (n_utts, S) of frames ``x`` (T, D) on the selection ``idx`` (T, C): the mean over an utterance's
    frames of log sum_{c in idx[t]} w_c N(x_t; means[s, c], variances[c]); 0 for an empty utterance."""
    x = np.asarray(x, dtype=np.float64)
    w, var, mu = (np.asarray(a, dtype=np.float64) for a in (weights, variances, means))
    idx = np.asarray(idx, dtype=np.int64)
    xs = x[:, None, :]                                     # (T, 1, D)
    v = var[idx]                                           # (T, C, D)
    base = np.log(w[idx]) - 0.5 * (x.shape[1] * np.log(2 * np.pi) + np.log(v).sum(axis=2))
    frame = np.empty((mu.shape[0], x.shape[0]))
    for s in range(mu.shape[0]):
        lp = base - 0.5 * (((xs - mu[s][idx]) ** 2) / v).sum(axis=2)
        m = lp.max(axis=1)
        frame[s] = m + np.log(np.exp(lp - m[:, None]).sum(axis=1))
    offs = np.asarray(frame_offsets, dtype=np.int64)
    out = np.zeros((len(offs) - 1, mu.shape[0]))
    for u in range(len(offs) - 1):
        if offs[u + 1] > offs[u]:
            out[u] = frame[:, offs[u] : offs[u + 1]].mean(axis=1)
    return out


def gpu_info(index: int) -> dict:
    """Read-only query of the card the numbers were taken on."""
    out = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=name,power.limit,clocks.max.sm",
                          "--format=csv,noheader,nounits"], capture_output=True, text=True, check=True).stdout
    name, power, clock = [s.strip() for s in out.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit_w": float(power), "sm_clock_max_mhz": float(clock)}


def stats(ms):
    return {"min": min(ms), "median": float(np.median(ms)), "max": max(ms), "reps": len(ms)}


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
        raise SystemExit("topc_bench.py measures the GPU kernels: no CUDA device found")
    import speech_signal_processing_b200 as ssp
    from speech_signal_processing_b200 import synth

    dev = torch.device("cuda", args.device)
    torch.cuda.set_device(dev)
    gpu = gpu_info(args.device)

    # ---- models and frames
    w, mu, var = synth.synth_ubm(K, D, seed=args.seed)
    means = np.concatenate([synth.synth_speaker_means(mu, N_SPK, seed=args.seed + 1, shift=0.25), mu[None]])
    sms = ssp.SharedModelSet(w, var, means, ref_model=-1, device=dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(args.seed)
    T = args.utts * UTT_FRAMES
    spk = torch.randint(0, N_SPK, (args.utts,), generator=gen, device=dev).repeat_interleave(UTT_FRAMES)
    comp = torch.multinomial(torch.as_tensor(w, device=dev), T, replacement=True, generator=gen)
    d_means = torch.as_tensor(means, device=dev, dtype=torch.float32)
    feats = (d_means[spk, comp] + torch.as_tensor(np.sqrt(var), device=dev, dtype=torch.float32)[comp]
             * torch.randn((T, D), generator=gen, device=dev, dtype=torch.float32)).contiguous()
    del spk, comp
    offs = np.arange(args.utts + 1, dtype=np.int64) * UTT_FRAMES

    # ---- timings, alternating the scorers call by call
    arms = {"exact": lambda: sms.score(feats, offs)}
    for c in C_VALUES:
        arms[f"top{c}"] = (lambda c=c: sms.score_top_c(feats, offs, c=c))
    sms.score_top_c(feats, offs, c=C_VALUES[0])          # builds the reference set and the (a, b) table
    ref = sms._topc[0]
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
    ubm = N_SPK

    def llr(scores):
        s = scores.cpu().numpy()
        return s[:, :ubm] - s[:, ubm : ubm + 1]

    exact = llr(outs["exact"][0])
    agree = {}
    for c in C_VALUES:
        got = llr(outs[f"top{c}"][0])
        agree[f"top{c}"] = {"decisions_equal": int((got.argmax(axis=1) == exact.argmax(axis=1)).sum()),
                            "utterances": int(args.utts), "max_abs_llr_diff": float(np.abs(got - exact).max())}

    # ---- float64 check of a seeded sample, on the GPU's own selection
    rs = np.random.RandomState(args.seed + 2)
    pick = np.sort(rs.choice(args.utts, size=min(args.check_utts, args.utts), replace=False))
    rows = np.concatenate([np.arange(u * UTT_FRAMES, (u + 1) * UTT_FRAMES) for u in pick])
    d_rows = torch.as_tensor(rows, device=dev)
    x = feats[d_rows].cpu().numpy()
    sub_offs = np.arange(len(pick) + 1, dtype=np.int64) * UTT_FRAMES
    check = {"utterances": int(len(pick))}
    for c in C_VALUES:
        idx, _ = ref.top_components(feats, whole, c)
        want = reference_top_c(x, sub_offs, w, var, means, idx[d_rows].cpu().numpy())
        got = outs[f"top{c}"][0].cpu().numpy()[pick]
        check[f"top{c}"] = {"max_rel_score_err": float((np.abs(got - want) / np.maximum(1.0, np.abs(want))).max()),
                            "max_abs_llr_err": float(np.abs((got[:, :ubm] - got[:, ubm:]) - (want[:, :ubm] - want[:, ubm:])).max())}
    res = {
        "bench": "topc",
        "gpu": gpu,
        "shape": {"utterances": args.utts, "frames": T, "K": K, "D": D, "models": N_SPK + 1},
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
