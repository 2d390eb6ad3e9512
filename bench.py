#!/usr/bin/env python
"""bench.py -- frames/sec of MFCC + GMM-UBM scoring (1024 components) on B200.

    python bench.py --gpus N --steps K --warmup W        # this repo's CUDA path
    python bench.py --impl reference ...                  # the reference's CPU path (oracle port + sklearn)
    python bench.py ... --dump-outputs DIR                # also save the last timed step's scores and decisions

Headline workload (BASELINE.json configs[3], the one the metric is quoted on): per GPU, 10 000 test utterances of 3 s @
16 kHz int16 -> 39-d MFCC+delta+delta-delta with per-utterance CMVN (298 frames each, 2.98 M frames) -> scored against
1 000 MAP-enrolled speaker models + the UBM (1 001 models x 1 024 diagonal components) -> LLR argmax per utterance.
One "step" = one pass over that batch.  Multi-GPU: every rank owns its own batch of utterances, all models replicated,
no data-path collective (weak scaling); `strong` reports the fixed-size job (10 000 utterances in total) beside it.

Audio, models and checks
    One counter-based generator (`synth.synth_pcm_torch`) makes every utterance of every arm: a pure function of
    (speaker, utterance, sample), so the GPU arm (on the device), the CPU arm and the oracle check (on the host) see the
    same audio.  Speakers are real classes of that audio: the UBM is EM-trained on the enrolment features, the 1 000
    speaker models are mean-only relevance-MAP adaptations (r = 16) from 10 enrolment utterances each, and test
    utterance j belongs to speaker j mod 1000.
    `check.oracle_*`: OUTSIDE the timed region, the first `--oracle-utts` test utterances go through the float64 CPU leg
    (oracle front-end + oracle.gmm.score against all 1 001 models, GMM_UBM.py:191-197) and are compared with what the
    timed GPU path produced for them.

`value`  = frames/s with the PCM already resident in HBM (front-end kernel + scoring kernels + argmax).
`e2e`    = frames/s through the public host-to-host call `ssp.identify_pcm` from pinned HOST PCM (H2D copy inside the
           timed region, its tail overlapped with the kernels of the head part) to the decisions read back on the host.
`roofline` = the tcgen05 scoring kernel against the tensor roofline: algorithmic 4*D*K FLOP per (frame, model) / its
           CUDA-event time / the measured dense rate of the pipe it issues on -- kind::f16 for the shared-variance kernel
           (MEASURED_PEAKS.json bf16_tflops_sustained), kind::tf32 for the general one (profiles/tf32_peak.json);
           `frac_hw` = the same against SM clock x FLOP/clk/SM x SMs at the clock the run actually held; `mufu` = the
           exponentials of the log-sum-exp against the MUFU rate, the resource that actually binds.
`secondary` = BASELINE.json configs[1], [2], [4] (front-end throughput, frame-sharded UBM EM with its all-reduce
           isolated, 2048-component sweep), each with its own roofline and -- at N = 1 -- CPU baseline on a stated sample.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "frames/sec MFCC+GMM-UBM scoring (1024 comp)"
UNIT = "frames/s"
K_COMP, N_SPK, N_UTT, UTT_SAMPLES, DIM = 1024, 1000, 10000, 48000, 39
FRAMES_PER_UTT = 298
ENROL_UTTS, TEST_UTT_BASE = 10, 100     # utterance ids 0..9 of a speaker enrol it, ids >= 100 are test material
N_SMS, TF32_FLOP_PER_CLK_SM = 148, 4096  # kind::tf32: half the 8192 dense bf16 FLOP/clk/SM
FP32_FLOP_PER_CLK_SM = 256               # 128 FMA lanes
FRONTEND_FLOP_PER_FRAME = 17000.0        # DESIGN.md 4.2: FFT-dominated FP32 work per 25 ms frame (SURVEY: 15-20 k)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--utts", type=int, default=N_UTT, help="test utterances per GPU (default = the named config)")
    ap.add_argument("--speakers", type=int, default=N_SPK)
    ap.add_argument("--components", type=int, default=K_COMP)
    ap.add_argument("--precision", default="tf32", choices=["tf32", "tf32x2", "tf32x3", "fp32"])
    ap.add_argument("--scorer", default="shared", choices=["shared", "general"],
                    help="shared: the shared-variance tensor kernel (mean-only MAP speakers keep the UBM's weights and "
                         "variances); general: the kernel for arbitrary model sets")
    ap.add_argument("--cpu-utts", type=int, default=0, help="reference arm: utterances per step (0 = auto-size)")
    ap.add_argument("--cpu-budget", type=float, default=100.0, help="reference arm: seconds of CPU work for the whole run")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the configs 2 / 3 / 5 legs")
    ap.add_argument("--secondary-scale", type=float, default=1.0, help="shrink the secondary legs (smoke runs)")
    ap.add_argument("--oracle-utts", type=int, default=32, help="utterances of the float64 CPU check (0 = skip)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write what the timed path returned in its last step to DIR/*.npy, to compare two builds")
    ap.add_argument("--oracle-check", default=None, help=argparse.SUPPRESS)   # internal: npz path -> float64 scores
    ap.add_argument("--cpu-legs", default=None, help=argparse.SUPPRESS)       # internal: CPU baselines of the secondary legs
    return ap.parse_args()


def workload_name(a):
    return (f"config4: {a.components}-comp {DIM}-d GMM-UBM identify, {a.utts} utts x {FRAMES_PER_UTT} frames (3 s @16 kHz) "
            f"per GPU vs {a.speakers} MAP speakers + UBM")


def test_ids(lo, hi, n_spk):
    """(speaker, utterance id) of global test utterances lo..hi-1: speaker j mod S, a fresh utterance id each round."""
    j = np.arange(lo, hi, dtype=np.int64)
    return j % n_spk, TEST_UTT_BASE + j // n_spk


def gen_pcm(spk, utt, device, n_samples=UTT_SAMPLES, chunk=500):
    """(len(spk) * n_samples,) int16 on `device` from the shared generator, built chunk by chunk."""
    import torch

    from speech_signal_processing_b200 import synth

    out = torch.empty(len(spk) * n_samples, dtype=torch.int16, device=device)
    for lo in range(0, len(spk), chunk):
        hi = min(len(spk), lo + chunk)
        out[lo * n_samples : hi * n_samples] = synth.synth_pcm_torch(spk[lo:hi], utt[lo:hi], n_samples, device).flatten()
    return out


# ------------------------------------------------------------------------------------------------
# CPU legs: the reference's own path (sidekit-recipe MFCC restatement + sklearn / oracle GMM maths)
# ------------------------------------------------------------------------------------------------
_W = {}


def _cpu_worker_init(w, mu, var):
    from threadpoolctl import threadpool_limits

    _W["lim"] = threadpool_limits(1)
    _W["params"] = (w, mu, var)


def _cpu_score_task(task):
    """score one feature matrix against a slice of speaker models with sklearn (GMM_UBM.py:194)."""
    from sklearn.mixture import GaussianMixture

    feat, lo, hi = task
    w, mu, var = _W["params"]
    out = np.empty(hi - lo)
    gm = GaussianMixture(n_components=len(w), covariance_type="diag")
    for i in range(lo, hi):
        gm.weights_, gm.means_, gm.covariances_ = w, mu[i], var
        gm.precisions_cholesky_ = 1.0 / np.sqrt(var)
        out[i - lo] = gm.score(feat)
    return lo, out


def _cpu_oracle_task(task):
    """float64 oracle scores (oracle/gmm.py restates sklearn _gaussian_mixture.py:536-553, _base.py:373,393)."""
    from oracle import gmm as ogmm

    feat, lo, hi = task
    w, mu, var = _W["params"]
    return lo, np.array([ogmm.score(feat, w, mu[i], var) for i in range(lo, hi)])


def _cpu_frontend_task(sig):
    from oracle import frontend as ofe

    return ofe.features(sig, preset="sidekit", delta_order=2, cmvn=True)


def cpu_models(a):
    """Model parameters for the CPU arm (values do not change its cost): synthetic UBM + shifted speaker means."""
    from speech_signal_processing_b200 import synth

    w, mu, var = synth.synth_ubm(a.components, DIM, seed=0)
    return w, np.concatenate([synth.synth_speaker_means(mu, a.speakers, seed=1, shift=0.25), mu[None]]), var


def run_reference(a):
    """Times GMM_UBM.py's per-utterance recipe on the host cores: extract_feature (:89-93, sidekit restatement + delta x2
    + scale) then GMM[i].score(x) - UBM.score(x) for every model (:191-197), on a bounded sample of the workload's
    utterances per step (the same generator the GPU arm uses, the first utterances of rank 0's batch), all cores busy."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from concurrent.futures import ProcessPoolExecutor

    cores = os.cpu_count() or 1
    procs = max(1, min(cores, 64))
    w, means, var = cpu_models(a)
    n_models = a.speakers + 1

    def pcm_of(n):
        spk, utt = test_ids(0, n, a.speakers)
        return gen_pcm(spk, utt, "cpu").numpy().reshape(n, UTT_SAMPLES)

    with ProcessPoolExecutor(procs, initializer=_cpu_worker_init, initargs=(w, means, var)) as pool:
        # calibrate: one utterance against 2 models per worker
        sig0 = pcm_of(1)[0]
        t0 = time.perf_counter()
        f0 = _cpu_frontend_task(sig0)
        list(pool.map(_cpu_score_task, [(f0, i % (n_models - 1), i % (n_models - 1) + 2) for i in range(0, 2 * procs, 2)]))
        per_pair = (time.perf_counter() - t0) / 2.0  # wall seconds per (utt, model) per worker
        budget = a.cpu_budget / max(1, a.steps + a.warmup)   # whole run within a few minutes
        n_utt = a.cpu_utts or int(max(1, min(64, budget / max(1e-6, per_pair * n_models / procs))))
        sigs = list(pcm_of(n_utt))
        chunk = max(1, (n_models + procs - 1) // procs)

        def step():
            feats = list(pool.map(_cpu_frontend_task, sigs))
            tasks = [(f, lo, min(lo + chunk, n_models)) for f in feats for lo in range(0, n_models, chunk)]
            pred = np.zeros((n_utt, n_models))
            per_utt = (n_models + chunk - 1) // chunk
            for j, (lo, out) in enumerate(pool.map(_cpu_score_task, tasks)):
                pred[j // per_utt, lo : lo + len(out)] = out
            return (pred[:, :-1] - pred[:, -1:]).argmax(axis=1), sum(len(f) for f in feats)

        for _ in range(a.warmup):
            step()
        t0 = time.perf_counter()
        frames = 0
        for _ in range(a.steps):
            _, nf = step()
            frames += nf
        dt = time.perf_counter() - t0
    val = frames / dt
    sample = (f"the first {n_utt} of {a.utts} test utterances per step (same generator as the GPU arm) x all {a.speakers}+1 "
              f"models, {procs} worker processes (1 BLAS thread each)")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1e3 * dt / a.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(a), "sample": sample},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": procs, "kind": "port", "sample": sample,
                         "host_cpu_count": cores},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def run_oracle_check(path):
    """Internal (--oracle-check): float64 CPU scores for the utterances in `path` (npz: pcm (n, samples) int16, w, var,
    means (S+1, K, D) with the UBM last, gpu_feats of the first utterances) -> JSON on stdout."""
    from concurrent.futures import ProcessPoolExecutor

    z = np.load(path)
    pcm, w, var, means = z["pcm"], z["w"], z["var"], z["means"]
    gpu_feats = z["gpu_feats"]
    n_models = means.shape[0]
    procs = max(1, min(os.cpu_count() or 1, 64))
    chunk = max(1, (n_models + procs - 1) // procs)
    per_utt = (n_models + chunk - 1) // chunk
    t0 = time.perf_counter()
    with ProcessPoolExecutor(procs, initializer=_cpu_worker_init, initargs=(w, means, var)) as pool:
        feats = list(pool.map(_cpu_frontend_task, list(pcm)))
        n_same = gpu_feats.shape[0] // feats[0].shape[0]
        mats = feats + [gpu_feats[i * feats[0].shape[0] : (i + 1) * feats[0].shape[0]].astype(np.float64) for i in range(n_same)]
        tasks = [(f, lo, min(lo + chunk, n_models)) for f in mats for lo in range(0, n_models, chunk)]
        scores = np.zeros((len(mats), n_models))
        for j, (lo, out) in enumerate(pool.map(_cpu_oracle_task, tasks)):
            scores[j // per_utt, lo : lo + len(out)] = out
    feat_err = max(float(np.abs(feats[i] - mats[len(feats) + i]).max()) for i in range(n_same)) if n_same else None
    print(json.dumps({"scores": scores[: len(feats)].tolist(), "scores_on_gpu_feats": scores[len(feats) :].tolist(),
                      "feat_max_abs_err": feat_err, "seconds": time.perf_counter() - t0, "cores": procs}), flush=True)


def run_cpu_legs(a):
    """Internal (--cpu-legs): CPU baselines of the secondary configs on stated samples, all host cores -> JSON."""
    from concurrent.futures import ProcessPoolExecutor

    from sklearn.mixture import GaussianMixture

    cores = os.cpu_count() or 1
    procs = max(1, min(cores, 64))
    out = {}
    # config 2: oracle front-end (sidekit restatement + delta x2 + scale, GMM_UBM.py:89-93), one utterance per task
    n2 = 4 * procs
    spk, utt = test_ids(0, n2, 1000)
    sigs = list(gen_pcm(spk, utt, "cpu").numpy().reshape(n2, UTT_SAMPLES))
    with ProcessPoolExecutor(procs, initializer=_cpu_worker_init, initargs=(None, None, None)) as pool:
        list(pool.map(_cpu_frontend_task, sigs[:procs]))
        t0 = time.perf_counter()
        frames = sum(len(f) for f in pool.map(_cpu_frontend_task, sigs))
        dt = time.perf_counter() - t0
    out["config2"] = {"value": frames / dt, "unit": "frames/s", "cores": procs, "kind": "port",
                      "sample": f"{n2} of 100000 utterances, oracle sidekit-recipe front-end + delta x2 + scale, {procs} processes"}
    # config 3: sklearn EM (GMM_UBM.py:169-170) from fixed initial parameters, BLAS / OpenMP on all cores
    n3, k3, iters = 200_000, 512, 2
    x = synth_em_frames(n3, "cpu").numpy()
    rs = np.random.RandomState(0)
    gm = GaussianMixture(n_components=k3, covariance_type="diag", weights_init=np.full(k3, 1.0 / k3),
                         means_init=x[rs.choice(n3, k3, replace=False)].astype(np.float64),
                         precisions_init=np.tile(1.0 / x.var(axis=0).astype(np.float64), (k3, 1)), max_iter=iters, tol=0.0)
    import warnings

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        t0 = time.perf_counter()
        gm.fit(x)
        dt = time.perf_counter() - t0
    out["config3"] = {"value": n3 * iters / dt, "unit": "frames/s per EM iteration", "ms_per_iteration_per_M_frames": 1e3 * dt / iters / (n3 / 1e6),
                      "cores": cores, "kind": "reference",
                      "sample": f"sklearn {iters} EM iterations (+ final E-step) on {n3} of 36 M frames, K = 512, float32 input, BLAS threads = all cores"}
    # config 5: sklearn score, K = 2048, one utterance per length
    from speech_signal_processing_b200 import synth

    w, mu, var = synth.synth_ubm(2048, DIM, seed=0)
    gm = GaussianMixture(n_components=2048, covariance_type="diag")
    gm.weights_, gm.means_, gm.covariances_, gm.precisions_cholesky_ = w, mu, var, 1.0 / np.sqrt(var)
    tot_f, tot_t = 0, 0.0
    for secs in (1, 3, 10, 30):
        t = (secs * 16000 - 400) // 160 + 1
        xx = np.random.RandomState(secs).standard_normal((t, DIM))
        gm.score(xx[:50])
        t0 = time.perf_counter()
        gm.score(xx)
        tot_t += time.perf_counter() - t0
        tot_f += t
    out["config5"] = {"value": tot_f / tot_t, "unit": "frames/s per model", "cores": cores, "kind": "reference",
                      "sample": "sklearn GaussianMixture.score, K = 2048, one utterance each of 1 / 3 / 10 / 30 s, one model"}
    print(json.dumps(out), flush=True)


def synth_em_frames(n, device, seed=0):
    """config 3 frames: 64 true Gaussian clusters in 39-d (SURVEY 8(d)), float32 on `device`."""
    import torch

    from speech_signal_processing_b200 import synth

    w, mu, var = synth.synth_ubm(64, DIM, seed=0)
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    x = torch.empty((n, DIM), dtype=torch.float32, device=device)
    t_mu = torch.as_tensor(mu, device=device, dtype=torch.float32)
    t_sd = torch.as_tensor(np.sqrt(var), device=device, dtype=torch.float32)
    for lo in range(0, n, 1 << 22):
        hi = min(n, lo + (1 << 22))
        comp = torch.randint(0, 64, (hi - lo,), generator=g, device=device)
        x[lo:hi] = t_mu[comp] + t_sd[comp] * torch.randn((hi - lo, DIM), generator=g, device=device)
    return x


def _child_json(argv, timeout):
    out = subprocess.run([sys.executable, os.path.abspath(__file__)] + argv, capture_output=True, text=True, timeout=timeout,
                         env={**os.environ, "RANK": "0", "WORLD_SIZE": "1", "CUDA_VISIBLE_DEVICES": ""})
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    if not lines:
        raise RuntimeError((out.stderr or out.stdout)[-400:])
    return json.loads(lines[-1])


def cpu_baseline_subprocess(a):
    """The oracle-port CPU baseline, run in a child BEFORE this process touches CUDA (it forks workers)."""
    try:
        return _child_json(["--impl", "reference", "--steps", "1", "--warmup", "1", "--cpu-budget", "30", "--utts", str(a.utts),
                            "--speakers", str(a.speakers), "--components", str(a.components)], 600)["cpu_baseline"]
    except Exception as e:  # the baseline is reported, never required
        return {"value": None, "unit": UNIT, "cores": None, "kind": "port", "sample": f"failed: {e!r}"[:300]}


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append([c.strip() for c in ln.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        pw = [float(r[2]) for r in self.rows if len(r) >= 7 and r[2].replace(".", "").isdigit()]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "power_w_max": max(pw) if pw else None}


def measured_peaks():
    """(dict, source): MEASURED_PEAKS.json (driver-written: HBM GB/s, bf16 TF/s) + profiles/tf32_peak.json (measured by
    benchmarks/measure_tf32_peak.py the same way), else the fallback of B200_PROFILING.md."""
    pk, src = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        pk, src = json.load(open(p)), "measured (MEASURED_PEAKS.json)"
    try:
        with open(os.path.join(ROOT, "profiles", "tf32_peak.json")) as f:
            t = json.load(f)
        pk["tf32_tflops"], pk["tf32_tflops_sustained"] = float(t["tf32_tflops"]), float(t["tf32_tflops_sustained"])
        pk["tf32_source"] = "measured (profiles/tf32_peak.json): torch.matmul TF32 8192^3, burst / sustained"
    except (OSError, KeyError, ValueError):
        pk["tf32_tflops"], pk["tf32_tflops_sustained"] = pk["bf16_tflops"] / 2.0, pk["bf16_tflops_sustained"] / 2.0
        pk["tf32_source"] = src + ": bf16 / 2 -- kind::tf32 MMAs issue at half the bf16 rate"
    return pk, src


class Bench:
    """Shared state of the B200 arm: device, communicator, helpers that time on the device and take max over ranks."""

    def __init__(self, a):
        import torch

        self.a, self.torch = a, torch
        self.rank, self.world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device(f"cuda:{self.local}")
        self.comm = None
        if self.world > 1:
            from speech_signal_processing_b200.dist import Comm

            self.comm = Comm("nccl")
        self.peaks, self.peak_src = measured_peaks()

    def barrier(self):
        if self.comm is not None:
            self.comm.barrier()
        self.torch.cuda.synchronize()

    def timed(self, fn, steps, warmup):
        """ms per step of fn(): warm-up, barrier + synchronize on both sides, CUDA events on the launching stream, max
        over ranks."""
        torch = self.torch
        for _ in range(warmup):
            fn()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1)) / steps

    def max_over_ranks(self, v):
        t = self.torch.tensor([float(v)], dtype=self.torch.float64, device=self.dev)
        if self.comm is not None:
            self.comm.allreduce_max(t)
        return float(t.item())

    def sum_over_ranks(self, v):
        t = self.torch.tensor([float(v)], dtype=self.torch.float64, device=self.dev)
        if self.comm is not None:
            self.comm.allreduce_sum(t)
        return float(t.item())


def build_models(b: Bench, fe):
    """UBM (EM on the enrolment features, K components, from fixed initial parameters) + S mean-only MAP speaker models,
    all on the device.  Returns (ubm GaussianMixture, w (K,), var (K, D), means (S + 1, K, D) with the UBM last)."""
    import warnings

    import speech_signal_processing_b200 as ssp

    torch, a = b.torch, b.a
    K, S = a.components, a.speakers
    spk = np.repeat(np.arange(S, dtype=np.int64), ENROL_UTTS)
    utt = np.tile(np.arange(ENROL_UTTS, dtype=np.int64), S)
    pcm = gen_pcm(spk, utt, b.dev)
    feats, foffs, _ = fe.extract_device(pcm, np.arange(len(spk) + 1, dtype=np.int64) * UTT_SAMPLES)
    del pcm
    n = feats.shape[0]
    pick = torch.as_tensor(np.random.RandomState(0).choice(n, K, replace=False), device=b.dev)
    gm = ssp.GaussianMixture(n_components=K, covariance_type="diag", weights_init=np.full(K, 1.0 / K),
                             means_init=feats[pick].cpu().numpy().astype(np.float64),
                             precisions_init=np.tile(1.0 / feats.var(dim=0).cpu().numpy().astype(np.float64), (K, 1)),
                             max_iter=4, tol=0.0)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        gm.fit(feats)
    seg = foffs[::ENROL_UTTS].copy()                       # one segment per speaker = its ENROL_UTTS utterances
    _, smu, _ = ssp.map_adapt(gm, (feats, seg), relevance=16.0, adapt=("means",))
    w = torch.as_tensor(gm.weights_, device=b.dev)
    var = torch.as_tensor(gm.covariances_, device=b.dev)
    means = torch.cat([smu, torch.as_tensor(gm.means_, device=b.dev)[None]])
    return gm, w, var, means


def oracle_check(b: Bench, pcm_dev, fe, gpu_scores, w, var, means, n_check):
    """Float64 CPU leg for the first n_check utterances of this rank's batch (child process, outside any timed region)
    against the scores the GPU path produced for them."""
    torch, a = b.torch, b.a
    S = a.speakers
    n_same = min(4, n_check)
    feats, foffs, _ = fe.extract_device(pcm_dev[: n_same * UTT_SAMPLES], np.arange(n_same + 1, dtype=np.int64) * UTT_SAMPLES)
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "check.npz")
        np.savez(path, pcm=pcm_dev[: n_check * UTT_SAMPLES].cpu().numpy().reshape(n_check, UTT_SAMPLES), w=w.cpu().numpy(),
                 var=var.cpu().numpy(), means=means.cpu().numpy(), gpu_feats=feats.cpu().numpy())
        res = _child_json(["--oracle-check", path], 900)
    ref = np.asarray(res["scores"])
    got = gpu_scores[:n_check].cpu().numpy()
    llr_ref, llr_got = ref[:, :S] - ref[:, S:], got[:, :S] - got[:, S:]
    top2 = np.sort(llr_ref, axis=1)[:, -2:]
    margin = top2[:, 1] - top2[:, 0]
    differ = llr_ref.argmax(axis=1) != llr_got.argmax(axis=1)
    same = np.asarray(res["scores_on_gpu_feats"])
    out = {
        "oracle_utts": int(n_check), "oracle_models": int(S + 1),
        "oracle_max_rel": float((np.abs(got - ref) / np.abs(ref)).max()),
        "oracle_max_llr_abs": float(np.abs(llr_got - llr_ref).max()),
        "oracle_decisions_equal": bool(not differ.any()), "oracle_decisions_differ": int(differ.sum()),
        "oracle_min_top2_margin": float(margin.min()),
        "oracle_margin_of_differing": [float(m) for m in margin[differ]][:8],
        "oracle_accuracy": float((llr_ref.argmax(axis=1) == test_ids(b.rank * a.utts, b.rank * a.utts + n_check, S)[0]).mean()),
        "oracle_feat_max_abs_err": res["feat_max_abs_err"],
        # scoring alone: float64 oracle on the features the GPU front-end produced
        "oracle_scoring_only_max_rel": float((np.abs(got[: len(same)] - same) / np.abs(same)).max()) if len(same) else None,
        "oracle_seconds": res["seconds"], "oracle_cores": res["cores"],
        "oracle": "oracle/frontend.py (sidekit recipe, float64) + oracle/gmm.py score, GMM_UBM.py:191-197; outside the timed region",
    }
    del torch
    return out


DUMP_BYTES = 64_000_000


def dump_outputs(path, scores, decisions):
    """--dump-outputs: the last timed step's per-utterance scores against every model (UBM last) and its LLR-argmax
    decisions, as float64 .npy files.  Where the scores exceed DUMP_BYTES, a fixed, seeded sample of utterances is kept;
    scores_rows.npy lists which."""
    os.makedirs(path, exist_ok=True)
    n, m = scores.shape
    dec = decisions.cpu().numpy().astype(np.float64)
    fit = (DUMP_BYTES - dec.nbytes) // (8 * (m + 1))   # a score row plus its index
    rows = np.arange(n) if fit >= n else np.sort(np.random.RandomState(0).choice(n, fit, replace=False))
    np.save(os.path.join(path, "decisions.npy"), dec)
    np.save(os.path.join(path, "scores.npy"), scores.cpu().numpy()[rows])
    np.save(os.path.join(path, "scores_rows.npy"), rows.astype(np.float64))


# ---------------------------------------------------------------------------------------------- secondary legs
def leg_config2(b: Bench, scale):
    """BASELINE configs[1]: MFCC+delta+delta-delta (39-d, CMVN) over 100 000 x 3 s utterances, sharded over the ranks."""
    import speech_signal_processing_b200 as ssp

    torch = b.torch
    n_total = max(b.world, int(100000 * scale))
    n_utts = n_total // b.world
    distinct = min(n_utts, 10000)                           # generated once, tiled: the kernel's work ignores content
    spk, utt = test_ids(b.rank * distinct, (b.rank + 1) * distinct, 1000)
    part = gen_pcm(spk, utt + 50, b.dev)
    pcm = part.repeat((n_utts + distinct - 1) // distinct)[: n_utts * UTT_SAMPLES].contiguous()
    del part
    offs = np.arange(n_utts + 1, dtype=np.int64) * UTT_SAMPLES
    fe = ssp.FrontEnd(ssp.sidekit_recipe(), delta_order=2, cmvn=True, device=b.dev)
    out = torch.empty((n_utts * FRAMES_PER_UTT, DIM), dtype=torch.float32, device=b.dev)
    ms = b.timed(lambda: fe.extract_device(pcm, offs, out=out), steps=5, warmup=3)
    frames = b.sum_over_ranks(n_utts * FRAMES_PER_UTT)
    bytes_per_frame = (2.0 * UTT_SAMPLES + 4.0 * DIM * FRAMES_PER_UTT) / FRAMES_PER_UTT   # SURVEY 8(d): 478 B/frame
    per_gpu_fps = frames / b.world / (ms * 1e-3)
    gbs = per_gpu_fps * bytes_per_frame / 1e9
    alu_peak = N_SMS * FP32_FLOP_PER_CLK_SM * b.peaks.get("sm_max_mhz", 1965.0) * 1e6
    alu_ceiling = alu_peak / FRONTEND_FLOP_PER_FRAME
    return {"workload": f"config2: MFCC+d+dd 39-d CMVN, {n_total} x 3 s utterances over {b.world} GPU(s)", "value": frames / (ms * 1e-3),
            "unit": "frames/s", "ms_per_step": ms, "steps": 5, "warmup": 3,
            "roofline": {"bound": "hbm", "kernel": "frontend512_kernel", "achieved": gbs, "peak": b.peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": gbs / b.peaks["hbm_gbs"], "bytes_per_frame": bytes_per_frame, "per": "GPU",
                         "alu_ceiling": {"flop_per_frame": FRONTEND_FLOP_PER_FRAME, "fp32_peak_tflops": alu_peak / 1e12,
                                         "frames_per_s": alu_ceiling, "frac": per_gpu_fps / alu_ceiling,
                                         "note": "the FP32-ALU ceiling binds before HBM (SURVEY 7): FFT-dominated work per frame"}}}


def leg_config3(b: Bench, scale):
    """BASELINE configs[2]: 512-component UBM EM on 36 M x 39-d frames SHARDED over the ranks (36 M / N each); one
    all-reduce of [N, F, S, loglik, n] (324 KB float64) per iteration, timed on its own with CUDA events."""
    import warnings

    import speech_signal_processing_b200 as ssp

    torch = b.torch
    n_total, k, iters = int(36_000_000 * scale), 512, 10
    n = n_total // b.world
    x = synth_em_frames(n, b.dev, seed=b.rank)
    # identical initial parameters on every rank: rank 0's first frames
    init = x[:k].clone()
    v0 = x[: 1 << 18].var(dim=0)
    if b.comm is not None:
        b.comm.broadcast(init, 0)
        b.comm.broadcast(v0, 0)
    kw = dict(n_components=k, covariance_type="diag", weights_init=np.full(k, 1.0 / k), means_init=init.cpu().numpy().astype(np.float64),
              precisions_init=np.tile(1.0 / v0.cpu().numpy().astype(np.float64), (k, 1)), tol=0.0, comm=b.comm)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ssp.GaussianMixture(max_iter=2, **kw).fit(x)   # warm-up (also sizes the workspace)
        gm = ssp.GaussianMixture(max_iter=iters, **kw)
        gm.allreduce_events = [] if b.comm is not None else None
        b.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        gm.fit(x)
        e1.record()
        b.barrier()
    ms = b.max_over_ranks(e0.elapsed_time(e1)) / iters
    ar_us = None
    if gm.allreduce_events:
        ar_us = b.max_over_ranks(1e3 * float(np.mean([s.elapsed_time(e) for s, e in gm.allreduce_events])))
    flop = 8.0 * DIM * k * n_total                      # SURVEY 8(d): logits + statistics, per iteration
    tf = flop / (ms * 1e-3) / 1e12
    peak = b.peaks["tf32_tflops_sustained"] * b.world
    mono = all(c >= p - 1e-4 for p, c in zip(gm.lower_bounds_, gm.lower_bounds_[1:]))
    return {"workload": f"config3: 512-comp UBM EM, {n_total} x 39-d frames sharded over {b.world} GPU(s), {iters} iterations",
            "value": n_total / (ms * 1e-3), "unit": "frames/s per EM iteration", "ms_per_iteration": ms, "iterations": iters,
            "allreduce": {"bytes": 8 * (k * (1 + 2 * DIM) + 2), "us_per_iteration": ar_us,
                          "note": "CUDA events around the NCCL all-reduce on the launching stream; includes the wait for the slowest rank"},
            "lower_bound_monotone": bool(mono), "lower_bound_last": float(gm.lower_bounds_[-1]),
            "roofline": {"bound": "tensor", "kernel": "gmm_em_lse_kernel + gmm_em_stats_kernel", "achieved": tf, "peak": peak, "unit": "TFLOP/s",
                         "frac": tf / peak, "flop": "algorithmic 8*D*K per frame per iteration", "peak_source": b.peaks["tf32_source"] + " (sustained x GPUs)"}}


def leg_config5(b: Bench, scale):
    """BASELINE configs[4]: 2048-component scoring vs frames per utterance (1-30 s), ~3 M frames in total sharded over the
    ranks, against the UBM alone and against 101 models."""
    import speech_signal_processing_b200 as ssp
    from speech_signal_processing_b200 import synth

    torch = b.torch
    k = 2048
    w, mu, var = synth.synth_ubm(k, DIM, seed=0)
    points = []
    # the single-pass rung streams FP16 images (kind::f16 MMAs) unless SSP_TC_TF32=1 forces the TF32 ones: the peak follows the pipe
    f16 = os.environ.get("SSP_TC_TF32", "0") != "1"
    peak5 = b.peaks["bf16_tflops_sustained"] if f16 else b.peaks["tf32_tflops_sustained"]
    for n_models in (1, 101):
        spk = np.concatenate([synth.synth_speaker_means(mu, n_models - 1, seed=1, shift=0.25), mu[None]]) if n_models > 1 else mu[None]
        ms_set = ssp.ModelSet(np.tile(w, (n_models, 1)), spk, np.tile(var, (n_models, 1, 1)), device=b.dev)
        for secs in (1, 2, 3, 5, 10, 20, 30):
            t = (secs * 16000 - 400) // 160 + 1
            n_utts = max(1, int(3_000_000 * scale) // t // b.world)
            total = n_utts * t
            x = torch.randn((total, DIM), device=b.dev)
            offs = np.arange(n_utts + 1, dtype=np.int64) * t
            ms = b.timed(lambda: ms_set.score(x, offs, precision="tf32"), steps=2, warmup=3 if secs == 1 else 1)
            frames = b.sum_over_ranks(total)
            tf = 4.0 * DIM * k * frames * n_models / (ms * 1e-3) / 1e12
            points.append({"seconds": secs, "frames_per_utt": int(t), "n_models": n_models, "ms": ms, "frames_per_s": frames / (ms * 1e-3),
                           "tflops": tf, "frac": tf / (peak5 * b.world)})
            del x
    best = max(p["tflops"] for p in points)
    full = [p for p in points if p["n_models"] == 101]
    return {"workload": f"config5: 2048-comp scoring sweep, 1-30 s utterances, ~{int(3_000_000 * scale)} frames over {b.world} GPU(s)",
            "value": float(np.mean([p["frames_per_s"] for p in full])), "unit": "frames/s (mean over lengths, 101 models)", "points": points,
            "roofline": {"bound": "tensor", "kernel": "gmm_score_tc_kernel", "achieved": best, "peak": peak5 * b.world,
                         "unit": "TFLOP/s", "frac": best / (peak5 * b.world),
                         "frac_of_tf32_peak": best / (b.peaks["tf32_tflops_sustained"] * b.world),
                         "flop": "algorithmic 4*D*K per (frame, model)",
                         "peak_source": ("MEASURED_PEAKS.json bf16_tflops_sustained (kind::f16 dense rate; FP16 operands, 11-bit significand as TF32)"
                                         if f16 else b.peaks["tf32_source"]) + " (sustained x GPUs)",
                         "note": "the exponentials of the log-sum-exp (2048 per frame and model) bind this kernel as they bind the headline one"}}


def run_b200(a):
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    cpu_base, cpu_legs = None, None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:   # children fork worker pools: before this process touches CUDA
        cpu_base = cpu_baseline_subprocess(a)
        if not a.no_secondary:
            try:
                cpu_legs = _child_json(["--cpu-legs", "all"], 600)
            except Exception as e:
                cpu_legs = {"error": f"{e!r}"[:300]}

    import torch

    import speech_signal_processing_b200 as ssp
    from speech_signal_processing_b200 import _lib

    b = Bench(a)
    dev, comm = b.dev, b.comm
    K, S, N, D = a.components, a.speakers, a.utts, DIM
    fe = ssp.FrontEnd(ssp.sidekit_recipe(), delta_order=2, cmvn=True, device=dev)
    # ---- models: UBM trained on the enrolment audio, speakers enrolled by MAP (means only, r = 16) from 10 utterances each
    ubm, w, var, means = build_models(b, fe)
    shared = a.scorer == "shared" and a.precision == "tf32"
    if shared:
        scorer = ssp.SharedModelSet(w, var, means, ref_model=S, device=dev)          # model S is the UBM
    else:
        scorer = ssp.ModelSet(w[None].expand(S + 1, -1), means, var[None].expand(S + 1, -1, -1), device=dev)
    # ---- test audio: this rank's slice of the global utterance list, in HBM and in pinned host memory
    spk_ids, utt_ids = test_ids(rank * N, (rank + 1) * N, S)
    pcm = gen_pcm(spk_ids, utt_ids, dev)
    host_pcm = torch.empty(N * UTT_SAMPLES, dtype=torch.int16, pin_memory=True)
    host_pcm.copy_(pcm)
    sample_offsets = np.arange(N + 1, dtype=np.int64) * UTT_SAMPLES
    host_dec = torch.empty(N, dtype=torch.int64, pin_memory=True)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    score_ms = []
    keep = {}

    def device_step(pcm_dev, offs=sample_offsets, timed=False):
        feats, foffs, _ = fe.extract_device(pcm_dev, offs)
        if timed:
            ev[2].record()
        scores, _ = scorer.score(feats, foffs, precision=a.precision)
        if timed:
            ev[3].record()
        keep["scores"] = scores
        llr = scores[:, :S] - scores[:, S:]
        return llr.argmax(dim=1), int(foffs[-1])

    def e2e_step():
        # the public host-to-host call: H2D of this step's PCM (the tail of the copy overlaps the kernels of the head),
        # front-end, scoring, LLR argmax, D2H of the decisions; returns once they have landed in host_dec
        _, nf = ssp.identify_pcm(host_pcm, sample_offsets, fe, scorer, ubm_index=S, precision=a.precision, out=host_dec)
        return nf

    for _ in range(a.warmup):
        device_step(pcm)
    b.barrier()
    sampler = ClockSampler(b.local)
    if rank == 0:
        sampler.start()
    lib = _lib.load()
    lib.ssp_reset_launch_count()
    # ---- timed region 1: inputs resident in HBM
    b.barrier()
    ev[0].record()
    frames = 0
    for _ in range(a.steps):
        dec, nf = device_step(pcm, timed=True)
        frames += nf
        torch.cuda.current_stream().synchronize()
        score_ms.append(ev[2].elapsed_time(ev[3]))
    ev[1].record()
    b.barrier()
    dev_ms = ev[0].elapsed_time(ev[1])
    launches = int(lib.ssp_launch_count())
    launch_log = _lib.launch_log()
    gpu_scores = keep["scores"]
    # ---- timed region 2: end to end from host buffers
    for _ in range(min(a.warmup, 2)):
        e2e_step()
    b.barrier()
    ev[0].record()
    for _ in range(a.steps):
        e2e_step()
    ev[1].record()
    b.barrier()
    e2e_ms = ev[0].elapsed_time(ev[1])
    clocks = sampler.stop() if rank == 0 else None
    # ---- the fixed-size job: N_total = a.utts utterances over ALL ranks (strong scaling of the named workload)
    n_strong = max(1, N // world)
    offs_strong = sample_offsets[: n_strong + 1]
    pcm_strong = pcm[: n_strong * UTT_SAMPLES]
    strong_ms = b.timed(lambda: device_step(pcm_strong, offs_strong), steps=3, warmup=1)
    strong_frames = b.sum_over_ranks(n_strong * FRAMES_PER_UTT)
    # host-to-host decisions vs HBM-resident decisions.  The two paths cut the batch differently, so the FP32 partial
    # sums inside a warp group other frames of an utterance (the cross-warp accumulation is float64): scores agree to
    # ~1e-6 absolute and a decision can only differ where the top-2 LLR margin is below that.
    e2e_dec = host_dec.to(dev)
    differ = (e2e_dec != dec).nonzero().flatten()
    e2e_check = {"utts": int(dec.numel()), "differ": int(differ.numel()), "largest_llr_margin_among_differing": 0.0}
    if differ.numel():
        llr = (gpu_scores[:, :S] - gpu_scores[:, S:])[differ]
        e2e_check["largest_llr_margin_among_differing"] = float(
            (llr.gather(1, dec[differ][:, None]) - llr.gather(1, e2e_dec[differ][:, None])).abs().max().item())
        del llr
    truth = torch.as_tensor(spk_ids, device=dev)
    accuracy = float((dec == truth).float().mean().item())

    dev_ms = b.max_over_ranks(dev_ms)
    e2e_ms = b.max_over_ranks(e2e_ms)
    total_frames = b.sum_over_ranks(frames)
    # ---- float64 CPU check of what the timed path produced (rank 0, outside the timed regions)
    check = {"e2e_vs_device_decisions": e2e_check, "planted_speaker_accuracy": accuracy}
    if rank == 0 and a.oracle_utts > 0:
        try:
            check.update(oracle_check(b, pcm, fe, gpu_scores, w, var, means, min(a.oracle_utts, N)))
        except Exception as e:
            check["oracle_error"] = f"{e!r}"[:300]
    if rank == 0 and a.dump_outputs:
        dump_outputs(a.dump_outputs, gpu_scores, dec)
    del gpu_scores
    keep.clear()

    # ---- secondary legs (all ranks take part)
    secondary = None
    if not a.no_secondary:
        del pcm, host_pcm, scorer
        torch.cuda.empty_cache()
        secondary = {}
        for name, leg in (("config2", leg_config2), ("config3", leg_config3), ("config5", leg_config5)):
            try:
                secondary[name] = leg(b, a.secondary_scale)
                if cpu_legs is not None:
                    secondary[name]["cpu_baseline"] = cpu_legs.get(name, cpu_legs)
            except Exception as e:  # a failing leg must not lose the headline
                secondary[name] = {"error": f"{e!r}"[:300]}
            torch.cuda.empty_cache()
    if rank != 0:
        return

    peaks = b.peaks
    n_models = S + 1
    flop_per_launch = 4.0 * D * K * (frames / a.steps) * n_models
    k_ms = float(np.mean(score_ms))
    achieved = flop_per_launch / (k_ms * 1e-3) / 1e12
    general_f16 = (not shared) and a.precision != "fp32" and os.environ.get("SSP_TC_TF32", "0") != "1"
    if shared or general_f16:
        # kind::f16 MMAs (FP16 operands, FP32 accumulation): that pipe's measured dense rate
        peak, bound = peaks["bf16_tflops_sustained"], "tensor"
        peak_note = ("MEASURED_PEAKS.json bf16_tflops_sustained (kind::f16: FP16 and BF16 operands run at the same dense rate; "
                     "sustained: the kernel is timed inside a long step)")
    elif a.precision != "fp32":
        peak, peak_note, bound = peaks["tf32_tflops_sustained"], peaks["tf32_source"] + " (sustained: the kernel is timed inside a long step)", "tensor"
    else:
        peak, peak_note, bound = 70.0, "nominal FP32 CUDA-core FMA peak (no measured figure)", "tensor"
    kernel = "gmm_score_sv_kernel" if shared else ("gmm_score_tc_kernel" if a.precision != "fp32" else "gmm_score_simt_kernel")
    sm_mhz = (clocks or {}).get("sm_mhz") or peaks.get("sm_max_mhz", 1965.0)
    flop_per_clk_sm = 2 * TF32_FLOP_PER_CLK_SM if (shared or general_f16) else TF32_FLOP_PER_CLK_SM   # kind::f16: twice the kind::tf32 rate
    hw_peak = N_SMS * flop_per_clk_sm * sm_mhz * 1e6 / 1e12
    roof_extra = {"frac_hw": achieved / hw_peak, "hw_peak": hw_peak,
                  "hw_peak_note": f"{N_SMS} SMs x {flop_per_clk_sm} FLOP/clk/SM x {sm_mhz:.0f} MHz (median SM clock of the timed region)"}
    if shared:
        # SURVEY 8(d): with the shared-variance shortcut the executed tensor work is smaller than the algorithmic 4DK:
        # per (frame, model) 2 * KS * Kp with KS = roundup(D + 2, 16); the common part (3 passes over roundup(2D + 2, 16))
        # once per 32 models and once more in the pre-pass
        ks, kq, kp = (D + 2 + 15) // 16 * 16, (2 * D + 2 + 15) // 16 * 16, (K + 63) // 64 * 64
        frames_step = frames / a.steps
        exec_flop = 2.0 * kp * frames_step * (ks * n_models + 3.0 * kq * (n_models / 32.0 + 1.0))
        ex = exec_flop / (k_ms * 1e-3) / 1e12
        # the resource that binds: one exponential per (frame, model, component); by default 10 of 16 column pairs go through
        # MUFU ex2 (16 per clock per SM), 6 through a degree-3 FMA-pipe polynomial (SSP_SV_POLY_PAIRS)
        exps = frames_step * n_models * kp
        mufu_peak = N_SMS * 16.0 * sm_mhz * 1e6
        on_mufu = 1.0 - int(os.environ.get("SSP_SV_POLY_PAIRS", "6")) / 16.0
        roof_extra.update({"executed_tflops": ex, "executed_frac": ex / peak, "executed_frac_hw": ex / hw_peak,
                           "frac_of_tf32_peak": achieved / peaks["tf32_tflops_sustained"],
                           "mufu": {"exponentials_per_launch": exps, "on_mufu": on_mufu, "mufu_per_s_peak": mufu_peak,
                                    "frac": on_mufu * exps / mufu_peak / (k_ms * 1e-3),
                                    "frac_if_all_on_mufu": exps / mufu_peak / (k_ms * 1e-3),
                                    "note": "MUFU ex2 time at the measured SM clock over the kernel time: the exponentials of the "
                                            "log-sum-exp (MUFU + FMA pipes + their issue slots), not the tensor pipe, bound this kernel"},
                           "note": "achieved = algorithmic 4*D*K FLOP per (frame, model) against the dense rate of the pipe the kernel "
                                   "uses (kind::f16, FP16 operands with TF32's 11-bit significand, FP32 accumulation); the "
                                   "shared-variance form executes 2*(D+2 padded to 48)*K per (frame, model) plus a 3-pass common "
                                   "part per 32 models; round 1 issued kind::tf32 and quoted the TF32 peak (frac_of_tf32_peak)"})
    # dram__bytes_read.sum + dram__bytes_write.sum of this kernel at this size, from a committed ncu --set full capture
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f).get(kernel)
        if t and (t["utts"], t["speakers"], t["components"]) == (N, S, K):
            traffic = {"bytes": t["dram_bytes"], "unit": "B per launch", "algorithmic_bytes": t.get("algorithmic_bytes"),
                       "source": t["source"]}
    except Exception:
        traffic = None
    line = {
        "metric": METRIC, "value": total_frames / (dev_ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": dev_ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": ("f16 operands (11-bit significand, as tf32) / f32 accumulate; common part 3-pass f32 grade" if shared else
                  {"tf32": "f16 operands (11-bit significand, as tf32) / f32 accumulate" if general_f16 else "tf32",
                   "tf32x2": "f16 operands, model operand as hi + lo (2 passes)" if general_f16 else "tf32 (2 passes)",
                   "tf32x3": "f16 hi + lo pieces of both operands (3 passes, f32 grade)" if general_f16 else "tf32 (3 passes)",
                   "fp32": "f32"}[a.precision]), "data": "synthetic",
        "config": {"workload": workload_name(a), "parallelism": f"utterances sharded x{world}, models replicated",
                   "l2": "inputs per step (0.96 GB PCM, 0.1-0.33 GB model tiles) exceed the 126 MB L2", "scorer": a.scorer,
                   "audio": "synth.synth_pcm_torch (counter-based; the CPU arm and the oracle check regenerate the same utterances)",
                   "models": "UBM: 4 EM iterations on the enrolment features; speakers: mean-only MAP (r = 16) from 10 utterances each",
                   "frames_x_models_per_s": total_frames * n_models / (dev_ms * 1e-3)},
        "e2e": {"value": total_frames / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(N * UTT_SAMPLES * 2),
                "d2h_bytes_per_step": int(N * 8), "ms_per_step": e2e_ms / a.steps},
        "strong": {"value": strong_frames / (strong_ms * 1e-3), "unit": UNIT, "total_utts": int(n_strong * world), "utts_per_gpu": int(n_strong),
                   "ms_per_step": strong_ms, "note": "the fixed-size job (config 4's 10 000 utterances in total) split over the ranks"},
        "gpu_launches": launches, "gpu_launch_log": launch_log,
        "roofline": {"bound": bound, "kernel": kernel, **roof_extra,
                     "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "traffic": traffic,
                     "kernel_ms": k_ms, "kernel_share_of_step": k_ms / (dev_ms / a.steps), "peak_source": peak_note,
                     "frac_of_bf16_peak": achieved / peaks["bf16_tflops_sustained"]},
        "clocks": clocks,
        "check": check,
    }
    if secondary is not None:
        line["secondary"] = secondary
    if cpu_base is not None:
        line["cpu_baseline"] = cpu_base
    print(json.dumps(line), flush=True)


def _shutdown():
    try:
        import torch.distributed as dist

        if dist.is_initialized():
            dist.destroy_process_group()
    except Exception:
        pass


if __name__ == "__main__":
    args = parse_args()
    if args.oracle_check:
        run_oracle_check(args.oracle_check)
    elif args.cpu_legs:
        run_cpu_legs(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)
        _shutdown()
