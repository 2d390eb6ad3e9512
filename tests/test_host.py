"""Host-side logic that needs no GPU: recipe tables, sharding, the N>1 reduction path over gloo,
and the guarantees that the product never routes through the oracle or a CPU fallback."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import speech_signal_processing_b200 as ssp
from oracle import frontend as ofe
from speech_signal_processing_b200 import dist as sdist
from speech_signal_processing_b200 import frontend as pfe
from speech_signal_processing_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_recipe_tables_match_oracle(golden):
    r = ssp.sidekit_recipe()
    assert (r.frame_len, r.frame_shift, r.nfft, r.framing, r.preemph_mode) == (400, 160, 512, 0, 1)
    np.testing.assert_allclose(r.fbank, ofe.sidekit_trfbank(16000, 512, 100, 8000, 0, 24)[0], atol=1e-15)
    np.testing.assert_allclose(r.dct, ofe.dct2_ortho_matrix(13, 24, first=1), atol=1e-15)
    np.testing.assert_allclose(r.window, np.hanning(400), atol=1e-15)
    p = ssp.psf_recipe()
    np.testing.assert_allclose(p.fbank, ofe.psf_filterbanks(), atol=1e-15)
    assert p.fbank.shape == (26, 257) and p.window.min() == 1.0 and p.energy_mode == 2
    # the 'processing' filterbank is pinned by the reference's own mfccInitFilterBanks output
    g = golden("processing_mfcc.npz")
    for fs, key in ((16000, "fbank_16k_512"), (8000, "fbank_8k_512")):
        two_sided = g[key]
        folded = pfe.processing_filterbank(fs, 512)
        x = np.abs(np.fft.fft(np.random.RandomState(0).standard_normal(512)))
        np.testing.assert_allclose(folded @ x[:257], two_sided @ x, rtol=1e-12)
    with pytest.raises(NotImplementedError):
        ssp.processing_recipe(16000, 5000, 160)
    # the drop-in of utils.processing.mfccInitFilterBanks itself (utils/processing.py:42-88), against its own output
    fb, freqs = ssp.mfccInitFilterBanks(16000, 512)
    np.testing.assert_allclose(fb, g["fbank_16k_512"], atol=1e-14)
    np.testing.assert_allclose(freqs, g["freqs_16k_512"], atol=1e-12)
    np.testing.assert_allclose(ssp.mfccInitFilterBanks(8000, 512)[0], g["fbank_8k_512"], atol=1e-14)


@pytest.mark.parametrize("fs,frame_size,step,tag", [(16000, 400, 160, "c"), (8000, 512, 256, "a"), (8000, 255, 100, None)])
def test_processing_tables_reproduce_reference_for_any_frame_size(golden, fs, frame_size, step, tag):
    """What the kernel computes from the 'processing' tables (window -> one-sided magnitude / nfft -> folded
    filterbank -> log10(. + 1e-8) -> DCT rows), emulated in numpy, against the unmodified utils/processing.py
    output; frame sizes that are not a power of two (nfft = frame length, utils/processing.py:129) and odd ones
    (bin nfft/2 has a mirror image then) included."""
    r = ssp.processing_recipe(fs, frame_size, step)
    assert r.nfft == frame_size and r.fbank.shape == (40, frame_size // 2 + 1)
    if tag is None:
        sig = synth.synth_utterance(2, 5, 3000, fs)
        want = ofe.processing_mfcc(sig, fs, frame_size, step)
    else:
        g = golden("processing_mfcc.npz")
        sig, want = g[f"{tag}_sig"], g[f"{tag}_mfcc"]
    n_frames = -(-len(sig) // step)
    padded = np.zeros((n_frames - 1) * step + frame_size)
    padded[: len(sig)] = sig
    frames = np.stack([padded[t * step : t * step + frame_size] for t in range(n_frames)]) * r.window
    spec = np.abs(np.fft.rfft(frames, r.nfft, axis=1)) * r.spec_scale
    got = np.log10(spec @ r.fbank.T + r.log_add) @ r.dct.T
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-9)


def test_librosa_recipe_tables_match_oracle():
    """Host tables of the librosa convention (MFCC_DTW.py:27-30) and the kernel's mirror-index rule, emulated in numpy."""
    r = ssp.librosa_recipe()
    assert (r.frame_len, r.frame_shift, r.nfft, r.framing, r.log_type, r.preemph_mode) == (2048, 512, 2048, 3, 3, 0)
    np.testing.assert_allclose(r.fbank, ofe.librosa_mel_filters(8000, 2048), atol=1e-14)
    np.testing.assert_allclose(r.extra["dct"], ofe.dct2_ortho_matrix(13, 128), atol=1e-15)
    assert ssp.librosa_recipe(pad_mode="constant").framing == 4 and ssp.librosa_recipe(center=False).framing == 0
    for n in (12000, 700, 2):  # 700 and 2: the padding folds more than once
        sig = synth.synth_utterance(3, n % 7, n, 8000).astype(np.float64)
        t_frames = 1 + n // 512
        idx = np.arange(t_frames)[:, None] * 512 + np.arange(2048)[None, :] - 1024
        per = 2 * (n - 1)
        m = np.mod(idx, per)
        m = np.where(m >= n, per - m, m)
        power = np.abs(np.fft.rfft(sig[m] * r.window, axis=1)) ** 2
        db = 10 * np.log10(np.maximum(power @ r.fbank.T, r.log_zero_floor))
        db = np.maximum(db, db.max() - r.extra["top_db"])
        np.testing.assert_allclose((db @ r.extra["dct"].T).T, ofe.librosa_mfcc(sig), atol=1e-8)
    with pytest.raises(NotImplementedError):
        ssp.librosa_recipe(pad_mode="edge")


def test_dct_rows_and_lifter():
    np.testing.assert_allclose(pfe.dct_rows(13, 26), ofe.dct2_ortho_matrix(13, 26), atol=1e-15)
    lift = 1 + 11 * np.sin(np.pi * np.arange(13) / 22)
    np.testing.assert_allclose(ssp.psf_recipe().dct, ofe.dct2_ortho_matrix(13, 26) * lift[:, None], atol=1e-14)


def test_shard_helpers():
    for n, w in [(10, 3), (7, 8), (10000, 8), (0, 2)]:
        spans = [sdist.shard_range(n, r, w) for r in range(w)]
        assert spans[0][0] == 0 and spans[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
        sizes = [b - a for a, b in spans]
        assert max(sizes) - min(sizes) <= 1
    lens = np.random.RandomState(1).randint(98, 2998, size=200)
    parts = sdist.shard_by_load(lens, 8)
    assert sorted(np.concatenate(parts).tolist()) == list(range(200))
    loads = [lens[p].sum() for p in parts]
    assert (max(loads) - min(loads)) <= lens.max()


def test_split_for_overlap_cuts_on_whole_waves():
    from speech_signal_processing_b200.ubm import _WAVE_FRAMES, split_for_overlap

    nfr = np.full(10000, 298)
    n = split_for_overlap(nfr)  # config 4: a tenth of 2.98 M frames = 7.9 waves -> 8 waves
    assert 0 < n < 10000
    assert n * 298 <= 8 * _WAVE_FRAMES < (n + 1) * 298
    assert split_for_overlap(np.full(100, 298)) == 0           # too small to pay
    assert split_for_overlap(np.array([10 * _WAVE_FRAMES])) == 0  # one utterance cannot be cut
    ragged = np.random.RandomState(0).randint(98, 2998, size=5000)
    m = split_for_overlap(ragged, 0.25)
    assert 0 < m < 5000 and ragged[:m].sum() <= round(0.25 * ragged.sum() / _WAVE_FRAMES) * _WAVE_FRAMES
    assert split_for_overlap(np.array([300, 300, 300]), 0.3, min_frames=0) == 0  # head would be empty: no split
    assert split_for_overlap(np.full(40, 115), 0.3, min_frames=0) == 12           # below one wave: the plain fraction


def test_product_never_imports_the_oracle_or_reference():
    pkg = os.path.join(ROOT, "speech_signal_processing_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), f
                assert "/root/reference" not in text, f


def test_only_tests_smoke_and_bench_touch_the_oracle():
    """The oracle is test infrastructure: outside tests/ only __graft_entry__.py (smoke) and bench.py (CPU baseline /
    reference arm) may import it; helper scripts under benchmarks/ and profiles/ must not."""
    allowed = {os.path.join(ROOT, "__graft_entry__.py"), os.path.join(ROOT, "bench.py")}
    for top in ("benchmarks", "profiles", "include", "speech_signal_processing_b200"):
        for dirpath, _, files in os.walk(os.path.join(ROOT, top)):
            for f in files:
                if f.endswith((".py", ".sh")):
                    text = open(os.path.join(dirpath, f)).read()
                    assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), os.path.join(dirpath, f)
    for f in os.listdir(ROOT):
        path = os.path.join(ROOT, f)
        if f.endswith(".py") and path not in allowed:
            assert not re.search(r"^\s*(from|import)\s+oracle\b", open(path).read(), flags=re.M), f
    # bench.py: the oracle appears only in the CPU legs (functions whose names start with _cpu_ / run_reference)
    bench = open(os.path.join(ROOT, "bench.py")).read()
    for m in re.finditer(r"^\s*from oracle import", bench, flags=re.M):
        head = bench[: m.start()]
        fn = re.findall(r"^def (\w+)", head, flags=re.M)[-1]
        assert fn.startswith("_cpu_") or fn == "run_reference", fn


def test_no_cpu_fallback_without_a_gpu():
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ssp.mfcc(np.zeros(16000, dtype=np.int16))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ssp.GaussianMixture(n_components=2).fit(np.zeros((10, 3)))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ssp.delta(np.zeros((10, 13)))


_WORKER = r"""
import os, sys
import numpy as np, torch
sys.path.insert(0, {root!r})
from speech_signal_processing_b200.dist import Comm, shard_range
from speech_signal_processing_b200 import synth
from oracle import gmm as ogmm
comm = Comm("gloo")
w, mu, var = synth.synth_ubm(16, 7, seed=5)
x = synth.sample_gmm(w, mu, var, 1001, seed=6).astype(np.float64)
lo, hi = shard_range(len(x), comm.rank, comm.world_size)
n, f, s, ll = ogmm.suff_stats(x[lo:hi], w, mu, var)
flat = torch.from_numpy(np.concatenate([n.ravel(), f.ravel(), s.ravel(), [ll, hi - lo]]))
comm.allreduce_sum(flat)
rn, rf, rs, rll = ogmm.suff_stats(x, w, mu, var)
ref = np.concatenate([rn.ravel(), rf.ravel(), rs.ravel(), [rll, len(x)]])
assert np.allclose(flat.numpy(), ref, rtol=1e-10, atol=1e-9), np.abs(flat.numpy() - ref).max()
# replicated M-step from the reduced statistics == unsharded M-step
k, d = 16, 7
a = flat.numpy()
w2, mu2, var2 = ogmm.m_step(a[:k], a[k:k + k * d].reshape(k, d), a[k + k * d:k + 2 * k * d].reshape(k, d))
w1, mu1, var1 = ogmm.m_step(rn, rf, rs)
assert np.allclose(mu1, mu2) and np.allclose(var1, var2) and np.allclose(w1, w2)
rows = torch.arange(hi - lo, dtype=torch.float64)[:, None] + 100.0 * comm.rank
full = comm.gather_rows(rows, [shard_range(len(x), r, comm.world_size)[1] - shard_range(len(x), r, comm.world_size)[0]
                               for r in range(comm.world_size)])
assert full.shape[0] == len(x)
assert full[:, 0].tolist() == list(range(501)) + [100.0 + i for i in range(500)]  # rank order, padding rows dropped
# uneven shards incl. an empty one (1 speaker on 2 ranks in map_enrol_sharded): rank 1 contributes nothing
one = [shard_range(1, r, comm.world_size) for r in range(comm.world_size)]
mine = torch.full((one[comm.rank][1] - one[comm.rank][0], 2, 3), 7.0 + comm.rank, dtype=torch.float64)
got = comm.gather_rows(mine, [b - a for a, b in one])
assert got.shape == (1, 2, 3) and float(got.sum()) == 7.0 * 6 + 6.0 * [c for c, (a, b) in enumerate(one) if b > a][0]
mx = torch.tensor([1.0 + comm.rank, 5.0 - comm.rank])
comm.allreduce_max(mx)
assert mx.tolist() == [2.0, 5.0]
b = torch.tensor([float(comm.rank)])
comm.broadcast(b, 0)
assert b.item() == 0.0
comm.barrier()
print("rank", comm.rank, "ok")
"""


def test_sharded_statistics_allreduce_gloo_world2(tmp_path):
    """N/F/S of frame shards all-reduced over gloo (world_size 2) == unsharded statistics; the M-step
    from the reduced tensor == the unsharded M-step (SURVEY 8(e): UBM EM)."""
    script = tmp_path / "worker.py"
    script.write_text(_WORKER.format(root=ROOT))
    port = 29600 + (os.getpid() % 300)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", LOCAL_RANK=str(r), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port),
                   CUDA_VISIBLE_DEVICES="")
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                                      text=True))
    outs = [p.communicate(timeout=180)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0, o
        assert f"rank {r} ok" in o


def test_bench_reference_arm_prints_contract_line():
    """bench.py --impl reference: one JSON line with the contract keys (tiny sizes)."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--speakers", "6", "--components", "16", "--cpu-utts", "2"], capture_output=True, text=True, timeout=300,
                         env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert out.returncode == 0, out.stderr[-2000:]
    import json

    line = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["impl"] == "reference" and line["unit"] == "frames/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["higher_is_better"] is True


def test_install_rebinds_the_reference_module_names():
    """INTEGRATION.md section 1: ssp.install() replaces exactly the names GMM_UBM.py:16-20,53 binds (no GPU needed to
    rebind; the GPU test test_install_runs_the_reference_call_pattern runs the call pattern through them)."""
    import types

    mod = types.ModuleType("GMM_UBM")
    mod.untouched = object()
    keep = mod.untouched
    assert ssp.install(mod) is mod
    assert mod.GaussianMixture is ssp.GaussianMixture and mod.delta is ssp.delta
    assert mod.preprocessing.scale is ssp.scale and callable(mod.mfcc) and callable(mod.plp)
    assert mod.untouched is keep
    import inspect

    assert list(inspect.signature(ssp.install).parameters) == ["gmm_ubm_module"]


def test_auto_precision_rule():
    from speech_signal_processing_b200.mixture import resolve_precision

    assert resolve_precision("auto", 64, 26) == "tf32x3"      # config 1: small models need the FP32-grade rung
    assert resolve_precision("auto", 1024, 39) == "tf32"      # config 4
    assert resolve_precision("auto", 2048, 39) == "tf32"      # config 5
    assert resolve_precision("auto", 1024, 40) == "fp32"      # contraction 2D + 2 > 80: CUDA cores
    assert resolve_precision("tf32x2", 8, 5) == "tf32x2"
    with pytest.raises(ValueError):
        resolve_precision("bf16", 8, 5)


def test_counter_based_audio_is_a_pure_function_of_its_ids():
    """bench.py's three consumers (GPU arm, CPU arm, oracle check) regenerate utterances independently: any batch split
    must give the same samples."""
    import torch

    from speech_signal_processing_b200 import synth

    a = synth.synth_pcm_torch([3, 3, 7, 11], [0, 1, 100, 5], 4000, "cpu")
    b = torch.cat([synth.synth_pcm_torch([3], [0], 4000, "cpu"), synth.synth_pcm_torch([3, 7, 11], [1, 100, 5], 4000, "cpu")])
    assert a.dtype == torch.int16 and a.shape == (4, 4000) and torch.equal(a, b)
    assert not torch.equal(a[0], a[1]) and int((a == 0).sum()) == 0
    rms = a.float().pow(2).mean(dim=1).sqrt()
    assert torch.all((rms > 2900) & (rms < 3100))
    sys.path.insert(0, ROOT)
    import bench

    spk, utt = bench.test_ids(0, 2500, 1000)
    assert spk[1234] == 234 and utt[1234] == bench.TEST_UTT_BASE + 1 and utt.min() >= bench.TEST_UTT_BASE > bench.ENROL_UTTS
    pcm = bench.gen_pcm(spk[:3], utt[:3], "cpu", n_samples=2000, chunk=2)
    assert torch.equal(pcm.reshape(3, 2000), synth.synth_pcm_torch(spk[:3], utt[:3], 2000, "cpu"))


def test_bench_dump_outputs_keeps_to_its_budget(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float64 files, every decision, all score rows when they fit and otherwise the same seeded
    sample of rows on every run."""
    import torch

    sys.path.insert(0, ROOT)
    import bench

    scores = torch.randn((40, 11), dtype=torch.float64)
    dec = torch.arange(40) % 10
    bench.dump_outputs(str(tmp_path / "all"), scores, dec)
    load = lambda d, name: np.load(str(tmp_path / d / f"{name}.npy"))  # noqa: E731
    assert all(load("all", f).dtype == np.float64 for f in ("scores", "decisions", "scores_rows"))
    assert np.array_equal(load("all", "scores"), scores.numpy()) and np.array_equal(load("all", "decisions"), dec.numpy())
    assert np.array_equal(load("all", "scores_rows"), np.arange(40))
    monkeypatch.setattr(bench, "DUMP_BYTES", 2000)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), scores, dec)
    rows = load("a", "scores_rows").astype(np.int64)
    assert 0 < len(rows) < 40 and (np.diff(rows) > 0).all() and np.array_equal(rows, load("b", "scores_rows"))
    assert np.array_equal(load("a", "scores"), scores.numpy()[rows]) and len(load("a", "decisions")) == 40
    assert sum(load("a", f).nbytes for f in ("scores", "decisions", "scores_rows")) <= 2000


# ------------------------------------------------------------------------------------------------
# batched WAV ingest (wavio.py) against scipy.io.wavfile.read, the reader the reference uses (utils/tools.py:45-47)
# ------------------------------------------------------------------------------------------------
def _write_wav_with_extra_chunks(path, rate, data, extensible=False):
    """A 16-bit PCM file with a LIST chunk of odd size before the data chunk (and optionally WAVE_FORMAT_EXTENSIBLE)."""
    import struct

    data = np.ascontiguousarray(data, dtype="<i2")
    ch = 1 if data.ndim == 1 else data.shape[1]
    if extensible:
        fmt = struct.pack("<HHIIHH", 0xFFFE, ch, rate, rate * 2 * ch, 2 * ch, 16) + struct.pack("<HHI", 22, 16, 0) + \
            struct.pack("<H", 1) + b"\x00\x00\x00\x00\x10\x00\x80\x00\x00\xaa\x00\x38\x9b\x71"
    else:
        fmt = struct.pack("<HHIIHH", 1, ch, rate, rate * 2 * ch, 2 * ch, 16)
    lst = b"INFOabc"  # 7 bytes: padded to 8
    body = b"WAVE" + b"fmt " + struct.pack("<I", len(fmt)) + fmt + b"LIST" + struct.pack("<I", len(lst)) + lst + b"\x00" + \
        b"data" + struct.pack("<I", data.nbytes) + data.tobytes()
    with open(path, "wb") as f:
        f.write(b"RIFF" + struct.pack("<I", len(body)) + body)


def test_read_wav_batch_equals_scipy(tmp_path):
    from scipy.io import wavfile

    import speech_signal_processing_b200 as ssp

    rs = np.random.RandomState(3)
    cases = []
    for i, (n, ch) in enumerate([(16000, 1), (1, 1), (0, 1), (4801, 2), (333, 1), (777, 3)]):
        sig = rs.randint(-32768, 32767, size=(n,) if ch == 1 else (n, ch)).astype(np.int16)
        p = tmp_path / f"a{i}.wav"
        if i in (1, 3, 4):
            _write_wav_with_extra_chunks(str(p), 8000 + i, sig, extensible=(i == 4))
        else:
            wavfile.write(str(p), 16000, sig)
        cases.append(p)
    batch = ssp.read_wav_batch(cases, threads=3)
    assert len(batch) == len(cases) and batch.sample_offsets[0] == 0
    utts = batch.utterances()
    for p, got, rate in zip(cases, utts, batch.rates):
        want_rate, want = wavfile.read(str(p))
        want = want[:, 0] if want.ndim == 2 else want
        assert rate == want_rate and got.dtype == np.int16 and np.array_equal(got, want)
    assert batch.sample_offsets[-1] == sum(len(u) for u in utts)
    # anything but 16-bit PCM is refused (load_data then reads the tree the reference's way)
    wavfile.write(str(tmp_path / "f32.wav"), 16000, rs.randn(100).astype(np.float32))
    with pytest.raises(ValueError):
        ssp.read_wav_batch([tmp_path / "f32.wav"])
    (tmp_path / "junk.wav").write_bytes(b"not a wav file at all")
    with pytest.raises(ValueError):
        ssp.read_wav_batch([tmp_path / "junk.wav"])


def test_load_data_walks_the_tree_like_the_reference(tmp_path, capsys):
    """x, y and label_encoder as GMM_UBM.load_data (GMM_UBM.py:24-50) builds them, through the batched reader and -- for a
    tree holding a float file -- through the per-file fallback."""
    from scipy.io import wavfile

    import speech_signal_processing_b200 as ssp
    from speech_signal_processing_b200 import ubm

    rs = np.random.RandomState(4)
    root = tmp_path / "ASR_GMM"
    for s in range(3):
        for ses in range(2):
            d = root / f"spk{s}" / f"ses{ses}"
            d.mkdir(parents=True)
            for u in range(2):
                wavfile.write(str(d / f"u{u}.wav"), 16000, rs.randint(-3000, 3000, size=400 + 10 * u).astype(np.int16))

    def reference_walk():
        x, y, enc = [], [], {}
        for num, spk in enumerate(os.listdir(root)):
            enc[spk] = num
            for ses in os.listdir(root / spk):
                for w in os.listdir(root / spk / ses):
                    x.append(wavfile.read(str(root / spk / ses / w))[1])
                    y.append(num)
        return x, y, enc

    ubm.label_encoder.clear()
    x, y = ssp.load_data(str(root))
    rx, ry, enc = reference_walk()
    assert y == ry and dict(ubm.label_encoder) == enc and len(x) == 12
    assert all(np.array_equal(a, b) for a, b in zip(x, rx))
    assert "Loading data..." in capsys.readouterr().out
    batch, y2 = ssp.load_batch(str(root))
    assert y2 == ry and all(np.array_equal(a, b) for a, b in zip(batch.utterances(), rx))
    wavfile.write(str(root / "spk0" / "ses0" / "u0.wav"), 16000, rs.randn(50).astype(np.float32))
    ubm.label_encoder.clear()
    x3, y3 = ssp.load_data(str(root))
    rx3, ry3, _ = reference_walk()
    assert y3 == ry3 and all(np.array_equal(a, b) for a, b in zip(x3, rx3))
    ubm.label_encoder.clear()


# ------------------------------------------------------------------------------------------------
# arithmetic of the FP16-operand scoring kernels, emulated in numpy (no GPU): why the shared-variance kernel stores speakers as
# differences from the reference and evaluates the common part in three FP16 passes (DESIGN.md 4.1)
# ------------------------------------------------------------------------------------------------
def test_fp16_operand_scheme_error_budget():
    from speech_signal_processing_b200 import synth

    rs = np.random.RandomState(7)
    k, d, t = 256, 39, 200
    w, mu, var = synth.synth_ubm(k, d, seed=5)
    spk = synth.synth_speaker_means(mu, 1, seed=6, shift=0.25)[0]
    x = synth.sample_gmm(w, mu, var, t, seed=8)
    log2e = 1.4426950408889634

    def h(a):      # round to FP16 (11-bit significand), keep float64 for the FP32-or-better accumulation of the tensor core
        return np.asarray(a, dtype=np.float16).astype(np.float64)

    def logits64(m):  # (t, k) in log2 units, float64
        p = 1.0 / var
        c = np.log(w) - 0.5 * (d * np.log(2 * np.pi) + (m * m * p).sum(1)) + 0.5 * np.log(p).sum(1)
        return ((x * x) @ (-0.5 * p).T + x @ (m * p).T + c) * log2e

    # ---- common part: A = [x^2, x], B = [-1/(2 var), mu_ref / var]; one pass vs three passes (A_hi.B_hi + A_lo.B_hi + A_hi.B_lo)
    a = np.concatenate([x * x, x], axis=1)
    b = np.concatenate([-0.5 / var, mu / var], axis=1) * log2e
    exact = a @ b.T
    a_hi, b_hi = h(a), h(b)
    a_lo, b_lo = h(a - a_hi), h(b - b_hi)
    one = a_hi @ b_hi.T
    three = one + a_lo @ b_hi.T + a_hi @ b_lo.T
    err1, err3 = np.abs(one - exact).max(), np.abs(three - exact).max()
    assert err1 > 5e-3            # an 11-bit pass alone moves a logit by ~1e-2: too much for posteriors or LLRs of small models
    assert err3 < 3e-7 * np.abs(exact).max()   # the three-pass form is FP32 grade (what is left is a_lo . b_lo ~ 2^-22): 4e-5 on |logit| <= 434
    # ---- per-speaker part: rounding (mu_s - mu_ref) / var instead of mu_s / var
    full = h(x) @ h(spk / var * log2e).T
    diff = h(x) @ h((spk - mu) / var * log2e).T
    err_full = np.abs(full - x @ (spk / var * log2e).T).max()
    err_diff = np.abs(diff - x @ ((spk - mu) / var * log2e).T).max()
    assert err_diff < 0.35 * err_full   # MAP-adapted means sit close to the UBM's: the same 11 bits cost several times less
    # ---- and the log-likelihood ratio of an utterance: common part exact enough to cancel, differences in one FP16 pass
    ck = (-0.5 * ((spk * spk - mu * mu) / var).sum(1)) * log2e
    l_ref = logits64(mu)
    l_spk_kernel = three + (np.log(w) - 0.5 * (d * np.log(2 * np.pi) + (mu * mu / var).sum(1)) - 0.5 * np.log(var).sum(1)) * log2e + diff + ck

    def lse2(l):
        m = l.max(1, keepdims=True)
        return (m[:, 0] + np.log2(np.exp2(l - m).sum(1)))

    llr_exact = (lse2(logits64(spk)) - lse2(l_ref)).mean() / log2e
    llr_kernel = (lse2(l_spk_kernel) - lse2(l_ref)).mean() / log2e
    assert abs(llr_kernel - llr_exact) < 1e-3   # SURVEY 8(c): LLR within 1e-3 absolute
