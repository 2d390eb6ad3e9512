"""A/B of the general tensor kernel's single-pass rung at config 5's shape (K = 2048, 101 models) against the 3-pass rung.
    python benchmarks/tc_ab.py"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.environ.get("GRAFT_REPO_ROOT", os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import speech_signal_processing_b200 as ssp  # noqa: E402
from speech_signal_processing_b200 import synth  # noqa: E402

k, d, n_models = 2048, 39, 101
w, mu, var = synth.synth_ubm(k, d, seed=0)
spk = np.concatenate([synth.synth_speaker_means(mu, n_models - 1, seed=1, shift=0.25), mu[None]])
ms = ssp.ModelSet(np.tile(w, (n_models, 1)), spk, np.tile(var, (n_models, 1, 1)))
t, n = 298, 10000
x = torch.randn((n * t, d), device="cuda")
offs = np.arange(n + 1, dtype=np.int64) * t
ref = None
for prec in ("tf32", "tf32x3"):
    for _ in range(2):
        out = ms.score(x, offs, precision=prec)[0]
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        out = ms.score(x, offs, precision=prec)[0]
    e1.record()
    torch.cuda.synchronize()
    ms_call = e0.elapsed_time(e1) / 3
    if prec == "tf32x3":
        ref = out
    else:
        first = out
    print(prec, round(ms_call, 2), "ms",
          round(4.0 * d * k * n * t * n_models / ms_call / 1e9, 1), "TFLOP/s algorithmic")
print("single pass vs 3 passes: max rel", float(((first - ref).abs() / ref.abs()).max()))
