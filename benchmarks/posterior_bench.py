"""Frame posteriors on one GPU: UBM alignment (predict_proba) and labelling (predict) of a large frame set, one JSON line.

    python benchmarks/posterior_bench.py [--seed 0] [--reps 5] [--warmup 1] [--device 0] [--frames 4194304]

Workloads (generated from the seed on the device; a 512-component, 39-dimensional UBM, the feature width of 13 MFCCs
with deltas and accelerations):
  A  2^22 frames, ``resp``: the (T, K) float32 posteriors every Baum-Welch / i-vector statistic starts from.  Timed with
     the frames' operand images already prepared (reuse, what an EM run or a ``stats`` call on the same frames leaves
     behind) and separately including the preparation pass.  Algorithmic bytes per frame: 4 D read + 4 K written; the
     GB/s is set against the HBM rate ``bench.py`` uses (MEASURED_PEAKS.json ``hbm_gbs`` when present, else the data-sheet
     figure, labelled as such).
  B  the same frames, labels only (``predict``): frames/s and algorithmic TFLOP/s at 2 (2D + 2) K per frame (the logit
     contraction; the three BF16 products of the FP32-grade form are not counted).
Each: ``ssp_gmm_posteriors`` through the C ABI on preallocated buffers, CUDA events over --reps calls after --warmup,
min / median / max.  Check and CPU baseline: sklearn 1.9 ``predict_proba`` / ``predict`` in float64 on a seeded sample
of --sample frames (all host cores), against the device outputs of those frames: max |gamma - float64|, largest row-sum
deviation, and label agreement on the frames whose float64 top-2 margin exceeds 1e-3.  Writes nothing to the tree.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

K, D = 512, 39
DATASHEET_HBM_GBS = 7700.0  # NVIDIA HGX B200 data sheet, per GPU
MARGIN = 1e-3
PROBA_ATOL, ROWSUM_ATOL = 1e-4, 2e-5  # the bounds tests/test_gpu_posteriors.py states


def gpu_info(index: int) -> dict:
    """Read-only query of the card the numbers were taken on."""
    out = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=name,power.limit,clocks.max.sm",
                          "--format=csv,noheader,nounits"], capture_output=True, text=True, check=True).stdout
    name, power, clock = [s.strip() for s in out.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit_w": float(power), "sm_clock_max_mhz": float(clock)}


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            pk = json.load(f)
        if "hbm_gbs" in pk:
            return float(pk["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return DATASHEET_HBM_GBS, "data sheet (NVIDIA HGX B200, per GPU)"


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


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--frames", type=int, default=1 << 22)
    ap.add_argument("--sample", type=int, default=20000)
    args = ap.parse_args()
    if args.reps < 5:
        ap.error("--reps must be at least 5")
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("posterior_bench.py measures the GPU kernels: no CUDA device found")
    from sklearn.mixture import GaussianMixture as SkGM

    import speech_signal_processing_b200 as ssp
    from speech_signal_processing_b200 import _lib, synth

    dev = torch.device("cuda", args.device)
    torch.cuda.set_device(dev)
    gpu = gpu_info(args.device)
    peak, peak_src = hbm_peak()

    # ---- model and frames
    w, mu, var = synth.synth_ubm(K, D, seed=args.seed, spread=1.0)
    gen = torch.Generator(device=dev)
    gen.manual_seed(args.seed)
    T = args.frames
    comp = torch.multinomial(torch.as_tensor(w, device=dev), T, replacement=True, generator=gen)
    feats = (torch.as_tensor(mu, device=dev, dtype=torch.float32)[comp]
             + torch.as_tensor(np.sqrt(var), device=dev, dtype=torch.float32)[comp]
             * torch.randn((T, D), generator=gen, device=dev, dtype=torch.float32)).contiguous()
    del comp
    ms = ssp.ModelSet(w, mu, var, device=dev)
    lib = _lib.load()
    offs = torch.as_tensor(np.array([0, T], dtype=np.int64), device=dev)
    ws_bytes = int(lib.ssp_gmm_posteriors_workspace_bytes(C.byref(ms.dims), T, 1))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    resp = torch.empty((T, K), dtype=torch.float32, device=dev)
    labels = torch.empty(T, dtype=torch.int64, device=dev)

    def call(out_resp, out_label, reuse):
        _lib.check(lib.ssp_gmm_posteriors(_lib.ptr(feats), _lib.ptr(offs), 1, T, _lib.ptr(ms.pack), C.byref(ms.dims),
                                          _lib.ptr(out_resp), _lib.ptr(out_label), None, _lib.ptr(ws), ws_bytes, reuse,
                                          _lib.stream_ptr()), "ssp_gmm_posteriors")

    call(resp, None, 0)  # prepares the images the reuse timings start from
    lib.ssp_reset_launch_count()
    a_reuse = time_events(torch, lambda: call(resp, None, 1), args.reps, args.warmup)
    a_launches = _lib.launch_log()
    a_prep = time_events(torch, lambda: call(resp, None, 0), args.reps, args.warmup)
    lib.ssp_reset_launch_count()
    b_reuse = time_events(torch, lambda: call(None, labels, 1), args.reps, args.warmup)
    b_launches = _lib.launch_log()

    bytes_per_frame = 4 * D + 4 * K
    flop_per_frame = 2 * (2 * D + 2) * K

    def gbs(t):
        return T * bytes_per_frame / (t["median"] / 1e3) / 1e9

    # ---- check and CPU baseline
    rs = np.random.RandomState(args.seed + 1)
    idx = np.sort(rs.choice(T, size=min(args.sample, T), replace=False))
    d_idx = torch.as_tensor(idx, device=dev)
    x = feats[d_idx].cpu().numpy().astype(np.float64)
    g_dev = resp[d_idx].cpu().numpy().astype(np.float64)
    l_dev = labels[d_idx].cpu().numpy()
    sk = SkGM(n_components=K, covariance_type="diag")
    sk.weights_, sk.means_, sk.covariances_ = w, mu, var
    sk.precisions_cholesky_ = 1.0 / np.sqrt(var)
    sk.precisions_ = 1.0 / var
    sk.n_features_in_ = D
    t0 = time.perf_counter()
    g_ref = sk.predict_proba(x)
    t_proba = time.perf_counter() - t0
    t0 = time.perf_counter()
    l_ref = sk.predict(x)
    t_pred = time.perf_counter() - t0
    wlp = np.sort(sk._estimate_weighted_log_prob(x), axis=1)
    ok = wlp[:, -1] - wlp[:, -2] > MARGIN
    check = {
        "frames": int(len(idx)),
        "max_abs_gamma_err": float(np.abs(g_dev - g_ref).max()),
        "max_row_sum_dev": float(np.abs(g_dev.sum(axis=1) - 1.0).max()),
        "margin_frames": int(ok.sum()),
        "labels_equal_on_margin_frames": bool((l_dev[ok] == l_ref[ok]).all()),
        "labels_equal_all": int((l_dev == l_ref).sum()),
    }
    res = {
        "bench": "posteriors",
        "gpu": gpu,
        "shape": {"frames": T, "K": K, "D": D},
        "hbm_peak_gbs": peak,
        "hbm_peak_source": peak_src,
        "A_resp": {
            "prepared_ms": a_reuse,
            "with_prep_ms": a_prep,
            "launches_prepared": a_launches,
            "bytes_per_frame": bytes_per_frame,
            "gbs_prepared": gbs(a_reuse),
            "hbm_fraction_prepared": gbs(a_reuse) / peak,
            "gbs_with_prep": gbs(a_prep),
            "hbm_fraction_with_prep": gbs(a_prep) / peak,
            "frames_per_s_prepared": T / (a_reuse["median"] / 1e3),
        },
        "B_labels": {
            "prepared_ms": b_reuse,
            "launches": b_launches,
            "frames_per_s": T / (b_reuse["median"] / 1e3),
            "flop_per_frame": flop_per_frame,
            "tflops": T * flop_per_frame / (b_reuse["median"] / 1e3) / 1e12,
        },
        "check": check,
        "cpu_baseline": {"impl": "sklearn 1.9 predict_proba / predict, float64", "frames": int(len(idx)),
                         "host_cores": os.cpu_count(), "predict_proba_s": t_proba, "predict_s": t_pred,
                         "predict_proba_frames_per_s": len(idx) / t_proba, "predict_frames_per_s": len(idx) / t_pred},
    }
    res["ok"] = (check["max_abs_gamma_err"] <= PROBA_ATOL and check["labels_equal_on_margin_frames"]
                 and check["max_row_sum_dev"] <= ROWSUM_ATOL)
    print(json.dumps(res))
    return 0 if res["ok"] else 1


if __name__ == "__main__":
    sys.exit(main())
