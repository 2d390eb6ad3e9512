"""Config-4-shaped timing of the shared-variance scoring kernel against the general tensor kernel.

    python benchmarks/prof_score_sv.py [n_utts] [n_speakers] [K]
"""
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import speech_signal_processing_b200 as ssp
from speech_signal_processing_b200 import synth

n_utts = int(sys.argv[1]) if len(sys.argv) > 1 else 2000
n_spk = int(sys.argv[2]) if len(sys.argv) > 2 else 1000
k = int(sys.argv[3]) if len(sys.argv) > 3 else 1024
general = os.environ.get("SV_COMPARE", "1") == "1"
d, t = 39, 298
dev = torch.device("cuda")
w, mu, var = synth.synth_ubm(k, d, seed=0)
spk = np.concatenate([synth.synth_speaker_means(mu, n_spk, seed=1, shift=0.25), mu[None]])
t_spk, t_var = torch.as_tensor(spk, device=dev), torch.as_tensor(var, device=dev)
labels = (torch.arange(n_utts, device=dev) % n_spk).repeat_interleave(t)
feats = synth.synth_features_torch(n_utts * t, d, t_spk[:n_spk], t_var, labels, seed=3, device=dev)
offs = np.arange(n_utts + 1, dtype=np.int64) * t
sms = ssp.SharedModelSet(w, var, t_spk)


def timed(fn, steps=3, warmup=2):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps, out


ms_sv, (a, _) = timed(lambda: sms.score(feats, offs))
flop = 4.0 * d * k * n_utts * t * (n_spk + 1)
res = {"n_utts": n_utts, "n_models": n_spk + 1, "K": k, "sv_ms": ms_sv, "sv_algorithmic_tflops": flop / ms_sv / 1e9,
       "sv_frames_per_s": n_utts * t / ms_sv * 1e3}
if general:
    gms = sms.expand()
    ms_g, (b, _) = timed(lambda: gms.score(feats, offs, precision="tf32"))
    a, b = a.cpu().numpy(), b.cpu().numpy()
    res.update({"general_ms": ms_g, "general_tflops": flop / ms_g / 1e9, "max_rel_diff": float(np.abs(a - b).max() / np.abs(b).max()),
                "decisions_equal": bool((a[:, :n_spk].argmax(1) == b[:, :n_spk].argmax(1)).all())})
print(json.dumps(res))
