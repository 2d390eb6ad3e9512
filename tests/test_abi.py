"""The C-ABI library builds, loads and exports every symbol include/ssp_b200.h declares.
No compute calls: runs without a GPU."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from speech_signal_processing_b200 import _lib, build

    build.build()  # no-op when up to date; nvcc cross-compiles sm_100a without a GPU
    return _lib.load()


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "ssp_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(ssp_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_exported(lib):
    names = declared_symbols()
    assert len(names) >= 14
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/ssp_b200.h but not exported"


def test_binding_covers_header(lib):
    from speech_signal_processing_b200 import _lib

    assert set(_lib.PROTOTYPES) == set(declared_symbols())
    assert lib.ssp_abi_version() == 1


def test_host_only_entry_points(lib):
    """Pure host helpers of the ABI: frame counting rules and pack sizing."""
    from speech_signal_processing_b200 import _lib

    def cfg(framing):
        return _lib.FrontendCfg(400, 160, 512, 24, 13, framing, 1, 0.97, 0, 1.0, 0, 0.0, 0.0, 1, 1, 2, 1, 0)

    c0, c1, c2 = cfg(0), cfg(1), cfg(2)
    # 1 s @ 16 kHz -> 98 frames (report/final.pdf p.5); psf 99+1; enframe ceil(N/step)
    assert lib.ssp_frontend_num_frames(C.byref(c0), 16000) == 98
    assert lib.ssp_frontend_num_frames(C.byref(c0), 48000) == 298
    assert lib.ssp_frontend_num_frames(C.byref(c0), 399) == 0
    assert lib.ssp_frontend_num_frames(C.byref(c1), 48000) == 299
    assert lib.ssp_frontend_num_frames(C.byref(c1), 10) == 1
    assert lib.ssp_frontend_num_frames(C.byref(c2), 48000) == 300
    assert lib.ssp_frontend_num_frames(C.byref(c2), 0) == 0
    assert lib.ssp_frontend_max_frames(C.byref(c0)) > 2998  # a 30 s utterance fits the fused kernel
    dft = cfg(0)
    dft.nfft = 400  # not a power of two: accepted, direct-DFT path
    assert lib.ssp_frontend_num_frames(C.byref(dft), 48000) == 298
    bad = cfg(0)
    bad.nfft = 320  # shorter than the frame
    assert lib.ssp_frontend_num_frames(C.byref(bad), 48000) == 0
    bad.nfft = 8192
    assert lib.ssp_frontend_num_frames(C.byref(bad), 48000) == 0
    d = _lib.GmmDims(1001, 1024, 39)
    nbytes = lib.ssp_gmm_pack_bytes(C.byref(d))
    assert nbytes >= 1001 * 1024 * (80 + 80 + 1) * 4  # tensor tiles + exact rows + constants
    assert lib.ssp_gmm_pack_bytes(C.byref(_lib.GmmDims(1, 16, 81))) == 0
    assert lib.ssp_gmm_pack_bytes(C.byref(_lib.GmmDims(0, 16, 13))) == 0


def test_null_arguments_fail_without_touching_the_gpu(lib):
    from speech_signal_processing_b200 import _lib

    d = _lib.GmmDims(1, 16, 13)
    assert lib.ssp_gmm_pack_models(None, None, None, C.byref(d), None, None) == -1
    assert b"null" in lib.ssp_last_error()
    assert lib.ssp_delta(None, 10, 13, 0, None, None) == -1


def test_library_has_no_hidden_tuning_switches():
    """The kernels' tuning choices are constants in the sources.  The only environment variable the library reads is
    SSP_SV_GROUP_MB (the L2 group size of shared-variance scoring, which tests use to reach the multi-launch path), and no
    SSP_ macro selects code at build time."""
    import glob

    names, directives = set(), []
    for path in sorted(glob.glob(os.path.join(ROOT, "speech_signal_processing_b200", "csrc", "*.cu*"))):
        text = open(path).read()
        calls = re.findall(r"\bgetenv\s*\(", text)
        literal = re.findall(r"\bgetenv\s*\(\s*\"([^\"]*)\"\s*\)", text)
        assert len(literal) == len(calls), f"{os.path.basename(path)}: getenv with a computed name"
        names.update(literal)
        directives += [(os.path.basename(path), d) for d in re.findall(r"^[ \t]*#[ \t]*(?:if|ifdef|ifndef|elif)\b.*\bSSP_\w*", text, flags=re.M)]
    assert names == {"SSP_SV_GROUP_MB"}
    assert directives == []


def test_header_is_plain_c(tmp_path):
    """The boundary is a C ABI: include/ssp_b200.h must compile as C99 (no C++ or torch types in the signatures) and a
    C translation unit that calls the host-only entry points must link against the library."""
    import shutil
    import subprocess

    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    src = tmp_path / "use_abi.c"
    src.write_text(
        '#include "ssp_b200.h"\n'
        "#include <stdio.h>\n"
        "int main(void) {\n"
        "  ssp_frontend_cfg c = {400, 160, 512, 24, 13, 0, 1, 0.97f, 0, 1.0f, 0, 0.0f, 0.0f, 1, 2, 2, 1, 0};\n"
        "  ssp_gmm_dims d = {1001, 1024, 39};\n"
        '  printf("%d %lld %lld\\n", ssp_abi_version(), (long long)ssp_frontend_num_frames(&c, 48000),\n'
        "         (long long)(ssp_gmm_pack_bytes(&d) > 0));\n"
        "  return ssp_frontend_batch(0, 0, 1, &c, 0, 0, 0, 0, 0, 0, 0, 1, 0, 0, 0) == SSP_EINVAL ? 0 : 1;\n"
        "}\n")
    inc = os.path.join(ROOT, "include")
    subprocess.check_call([gcc, "-std=c99", "-Wall", "-Werror", "-fsyntax-only", "-I", inc, str(src)])
    from speech_signal_processing_b200 import _lib

    exe = tmp_path / "use_abi"
    libdir = os.path.dirname(_lib.LIB_PATH)
    subprocess.check_call([gcc, "-std=c99", "-I", inc, str(src), "-o", str(exe), "-L", libdir, "-l:" + os.path.basename(_lib.LIB_PATH),
                           "-Wl,-rpath," + libdir])
    out = subprocess.run([str(exe)], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    assert out.stdout.split() == ["1", "298", "1"]


def test_host_framing_rule_equals_the_abi_rule(lib):
    """FrontEnd.frame_counts (vectorised, used to build frame_offsets) == ssp_frontend_num_frames for every framing mode
    (sidekit / psf / processing.py / librosa centred, reflect and zero padded)."""
    import numpy as np

    import speech_signal_processing_b200 as ssp
    from speech_signal_processing_b200 import _lib

    rs = np.random.RandomState(0)
    lens = np.concatenate([np.arange(0, 1300), rs.randint(0, 200000, size=500)])
    recipes = [ssp.sidekit_recipe(), ssp.psf_recipe(), ssp.processing_recipe(16000, 400, 160), ssp.processing_recipe(8000, 512, 256),
               ssp.librosa_recipe(), ssp.librosa_recipe(pad_mode="constant", n_fft=512, hop_length=128), ssp.librosa_recipe(center=False)]
    for r in recipes:
        fe = ssp.FrontEnd.__new__(ssp.FrontEnd)   # host-side rule only: no device needed
        fe.recipe = r
        got = fe.frame_counts(lens)
        cfg = _lib.FrontendCfg(r.frame_len, r.frame_shift, r.nfft, r.fbank.shape[0], r.dct.shape[0], r.framing, r.preemph_mode,
                               r.preemph, r.spec_type, r.spec_scale, r.log_type, r.log_add, r.log_zero_floor, r.energy_mode, 0, 2, 0, 0)
        want = np.array([lib.ssp_frontend_num_frames(C.byref(cfg), int(n)) for n in lens])
        assert (got == want).all(), (r.name, r.framing, lens[np.nonzero(got != want)[0][:5]])
        assert want[lens > 4096].min() > 0   # the configuration was accepted (0 would mean "rejected")
        # the fused single-pass kernel holds a 3 s utterance of every convention (librosa keeps 128 bands per frame)
        assert lib.ssp_frontend_max_frames(C.byref(cfg)) >= max(300, int(fe.frame_counts([3 * 16000])[0]) if r.name != "librosa" else 100)


def test_pack_sizes_follow_the_documented_layouts(lib):
    """Host-only size queries: the shared-variance pack is [Kp/64 tiles][4 + S images] of 64 x roundup(D + 2, 16) FP16 values
    + a 128-byte tail and accepts D <= 39 (shared-memory bound of gmm_score_sv_kernel); the general pack grows with the
    number of models and carries the FP16 images of the single-pass rung."""
    from speech_signal_processing_b200 import _lib

    def sv(s, k, d):
        return int(lib.ssp_gmm_shared_pack_bytes(C.byref(_lib.GmmDims(s, k, d))))

    assert sv(1001, 1024, 39) == 16 * (1001 + 4) * 64 * 48 * 2 + 128
    assert sv(3, 100, 13) == 2 * (3 + 4) * 64 * 16 * 2 + 128        # K padded to 128, D + 2 = 15 -> 16
    assert sv(3, 64, 26) == 1 * (3 + 4) * 64 * 32 * 2 + 128
    assert sv(3, 64, 40) == 0 and sv(3, 64, 0) == 0 and sv(0, 64, 13) == 0
    general = [int(lib.ssp_gmm_pack_bytes(C.byref(_lib.GmmDims(m, 1024, 39)))) for m in (1, 2, 101)]
    assert 0 < general[0] < general[1] < general[2]
    per_model = (general[2] - general[1]) / 99.0
    # per component: E-section (float2 x 40 + cst) + TF32 hi and lo tiles (80 floats each) + BF16 hi and lo images of the
    # statistics kernels (80 each, sets of <= 1024 models) + FP16 hi and lo tiles (80 halfs each)
    assert abs(per_model - 1024 * (40 * 8 + 4 + 2 * 80 * 4 + 2 * 80 * 2 + 2 * 80 * 2)) < 4096
    assert int(lib.ssp_gmm_pack_bytes(C.byref(_lib.GmmDims(1, 64, 81)))) == 0
