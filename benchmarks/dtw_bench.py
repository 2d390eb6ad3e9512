"""DTW template matching on one GPU: all-pairs distance matrices of MFCC_DTW.py-sized workloads, one JSON line out.

    python benchmarks/dtw_bench.py [--seed 0] [--reps 5] [--warmup 1] [--device 0]

Workloads (generated from the seed on the device):
  A  10 000 queries x 1 000 templates, 30-100 frames, dim 13, euclidean -- utils.processing.MFCC at 8 kHz (512 / 256)
     on 1-3 s words;
  B  2 000 x 1 000 flattened MFCC_lib sequences (13 coefficients x 16-47 frames): dim 1, 208-611 values, euclidean.
Per workload: time per ssp.dtw_matrix call (device inputs, float64 matrix back on the host) and per dtw_kernel launch
alone, both from CUDA events over --reps calls after --warmup, with min / median / max; cells/s (sum of n * m over the
pairs) and pairs/s from the kernel time; the FP32-ALU fraction from shapes (3 dim + 4 operations per cell: difference
and FMA per element, sqrt, two mins and an add, over 148 SMs x 128 lanes x 2 x the maximum SM clock); the float64
reference on a seeded sample of >= 200 pairs (max relative error, argmin agreement over the sampled templates), whose
time is also the CPU baseline (vectorised anti-diagonal numpy, one core).  Scripts under benchmarks/ do not import the
test oracle, so the float64 reference lives here (:func:`dtw_float64`); tests/test_dtw.py holds it equal to
``oracle.dtw``.  Writes nothing to the tree.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
from scipy.spatial.distance import cdist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    "A": dict(n_q=10000, n_r=1000, lo=30, hi=100, dim=13, dist="euclidean", sample=(8, 32)),
    "B": dict(n_q=2000, n_r=1000, lo=208, hi=611, dim=1, dist="euclidean", sample=(8, 25)),
}
SMS, LANES = 148, 128


def dtw_float64(x, y, dist):
    """DTW distance in float64: C = cdist(x, y, dist), then the warp-1 recurrence one anti-diagonal per numpy step."""
    C = cdist(x, y, dist)
    n, m = C.shape
    D0 = np.full((n + 1, m + 1), np.inf)
    D0[0, 0] = 0.0
    for s in range(n + m - 1):           # cells with i + j == s
        i = np.arange(max(0, s - m + 1), min(n, s + 1))
        j = s - i
        D0[i + 1, j + 1] = C[i, j] + np.minimum(D0[i, j], np.minimum(D0[i, j + 1], D0[i + 1, j]))
    return float(D0[n, m])


def gpu_info(index: int) -> dict:
    """Read-only query of the card the numbers were taken on."""
    out = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=name,power.limit,clocks.max.sm",
                          "--format=csv,noheader,nounits"], capture_output=True, text=True, check=True).stdout
    name, power, clock = [s.strip() for s in out.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit_w": float(power), "sm_clock_max_mhz": float(clock)}


def make_set(torch, gen, n, lo, hi, dim, dev):
    lens = torch.randint(lo, hi + 1, (n,), generator=gen, device=dev).cpu().numpy().astype(np.int64)
    offs = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(lens, out=offs[1:])
    feats = torch.randn((int(offs[-1]), dim), generator=gen, device=dev, dtype=torch.float32)
    return feats, offs


def time_events(torch, fn, reps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    return {"min": min(ms), "median": float(np.median(ms)), "max": max(ms), "reps": reps}


def run_workload(name, w, args, torch, dev, peak_ops):
    import speech_signal_processing_b200 as ssp
    from speech_signal_processing_b200 import _lib, dtw

    gen = torch.Generator(device=dev)
    gen.manual_seed(args.seed * 1000 + ord(name))
    Q = make_set(torch, gen, w["n_q"], w["lo"], w["hi"], w["dim"], dev)
    R = make_set(torch, gen, w["n_r"], w["lo"], w["hi"], w["dim"], dev)
    ql, rl = np.diff(Q[1]), np.diff(R[1])
    cells = float(ql.sum()) * float(rl.sum())
    pairs = w["n_q"] * w["n_r"]

    result = {}
    call = time_events(torch, lambda: result.__setitem__("d", ssp.dtw_matrix(Q, R, w["dist"], device=dev)), args.reps,
                       args.warmup)
    # the kernel alone: the launch dtw_matrix makes (the set with the shorter longest sequence in shared memory)
    lib = _lib.load()
    rows, cols = (R, Q) if ql.max() < rl.max() else (Q, R)
    d_row, d_col = torch.as_tensor(rows[1], device=dev), torch.as_tensor(cols[1], device=dev)
    out = torch.empty((len(rows[1]) - 1, len(cols[1]) - 1), dtype=torch.float32, device=dev)
    col_max = int(np.diff(cols[1]).max())

    def launch():
        _lib.check(lib.ssp_dtw_batch(_lib.ptr(rows[0]), _lib.ptr(d_row), len(rows[1]) - 1, _lib.ptr(cols[0]), _lib.ptr(d_col),
                                     len(cols[1]) - 1, w["dim"], dtw.METRICS[w["dist"]], col_max, _lib.ptr(out),
                                     _lib.stream_ptr()), "ssp_dtw_batch")

    lib.ssp_reset_launch_count()
    kern = time_events(torch, launch, args.reps, args.warmup)
    launches = _lib.launch_log()
    d = result["d"]
    k_s = kern["median"] / 1e3

    # float64 reference on a seeded sample of queries x templates (also the CPU baseline)
    rs = np.random.RandomState(args.seed + ord(name))
    qi = np.sort(rs.choice(w["n_q"], w["sample"][0], replace=False))
    ri = np.sort(rs.choice(w["n_r"], w["sample"][1], replace=False))
    qh, rh = Q[0].cpu().numpy().astype(np.float64), R[0].cpu().numpy().astype(np.float64)
    qs = [qh[Q[1][i]:Q[1][i + 1]] for i in qi]
    rss = [rh[R[1][j]:R[1][j + 1]] for j in ri]
    t0 = time.perf_counter()
    want = np.array([[dtw_float64(a, b, w["dist"]) for b in rss] for a in qs])
    cpu_s = time.perf_counter() - t0
    got = d[np.ix_(qi, ri)]
    rel = float((np.abs(got - want) / np.maximum(want, 1e-30)).max())
    sample_cells = float(ql[qi].sum()) * float(rl[ri].sum())
    ops_per_cell = 3 * w["dim"] + 4
    return {
        "shape": {k: w[k] for k in ("n_q", "n_r", "lo", "hi", "dim", "dist")},
        "cells": cells,
        "pairs": pairs,
        "call_ms": call,
        "kernel_ms": kern,
        "kernel_launches": launches,
        "cells_per_s": cells / k_s,
        "pairs_per_s": pairs / k_s,
        "ops_per_cell": ops_per_cell,
        "fp32_alu_fraction": cells * ops_per_cell / k_s / peak_ops,
        "check": {"pairs": int(len(qi) * len(ri)), "max_rel_err": rel,
                  "argmin_equal": bool((np.argmin(got, axis=1) == np.argmin(want, axis=1)).all()),
                  "matrix_finite": bool(np.isfinite(d).all())},
        "cpu_baseline": {"impl": "dtw_float64: anti-diagonal numpy (float64), one process", "pairs": int(len(qi) * len(ri)),
                         "seconds": cpu_s, "cells_per_s": sample_cells / cpu_s, "host_cores": os.cpu_count()},
    }


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--workloads", default="A,B")
    args = ap.parse_args()
    if args.reps < 5:
        ap.error("--reps must be at least 5")
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("dtw_bench.py measures the GPU kernels: no CUDA device found")
    dev = torch.device("cuda", args.device)
    torch.cuda.set_device(dev)
    gpu = gpu_info(args.device)
    peak_ops = SMS * LANES * 2 * gpu["sm_clock_max_mhz"] * 1e6
    res = {"bench": "dtw", "gpu": gpu, "fp32_peak_ops_per_s": peak_ops}
    for name in args.workloads.split(","):
        res[name] = run_workload(name, WORKLOADS[name], args, torch, dev, peak_ops)
    res["ok"] = all(res[n]["check"]["max_rel_err"] <= 2e-5 and res[n]["check"]["argmin_equal"]
                    and res[n]["check"]["matrix_finite"] for n in args.workloads.split(","))
    print(json.dumps(res))
    return 0 if res["ok"] else 1


if __name__ == "__main__":
    sys.exit(main())
