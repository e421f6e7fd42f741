"""CPU-only tests of the host side: constant builders (bit-identical with the reference's
buffers), integer bookkeeping (Python and C), the C-ABI library (loads, exports every declared
symbol, validates arguments without touching a GPU) and the drop-in module surface."""
import ctypes
import math
import os
import re
import warnings

import numpy as np
import pytest
import torch
from conftest import ROOT, assert_close
from golden_cases import MEL_FB

import audio_b200
import audio_b200.functional as F
import audio_b200.transforms as T
from audio_b200 import _bookkeeping as bk
from audio_b200 import _build, _lib


@pytest.fixture(scope="module")
def lib():
    _build.build()  # no-op when the .so is fresh
    return _lib.lib()


# ---------------- constants: bit-identical with the reference's buffers ------------------------
def test_constants_bit_identical(ref_cases):
    m = T.MelSpectrogram(16000, n_fft=1024, hop_length=256, n_mels=80)
    assert np.array_equal(m.mel_scale.fb.numpy(), ref_cases["mel_c2_fb"])
    assert np.array_equal(m.spectrogram.window.numpy(), ref_cases["mel_c2_window"])
    m = T.MelSpectrogram(22050, n_fft=2048, hop_length=512, n_mels=128, norm="slaney", mel_scale="slaney", f_max=8000.0)
    assert np.array_equal(m.mel_scale.fb.numpy(), ref_cases["mel_slaney2048_fb"])
    mf = T.MFCC(16000, n_mfcc=40, melkwargs=dict(n_fft=1024, hop_length=256, n_mels=80))
    assert np.array_equal(mf.dct_mat.numpy(), ref_cases["mfcc_dct"])
    r = T.Resample(44100, 16000, resampling_method="sinc_interp_kaiser")
    assert r.width == 17 and r.gcd == 100 and tuple(r.kernel.shape) == (160, 1, 475)
    assert np.array_equal(r.kernel.numpy(), ref_cases["rs_kaiser_kernel"])
    r = T.Resample(44100, 16000)
    assert np.array_equal(r.kernel.numpy(), ref_cases["rs_hann_kernel"])


@pytest.mark.parametrize("i", range(len(MEL_FB)))
def test_melscale_fbanks_librosa(librosa_melfb, i):
    c = MEL_FB[i]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        fb = F.melscale_fbanks(c["n_fft"] // 2 + 1, c["fmin"], c["fmax"], c["n_mels"], c["sample_rate"], c["norm"], c["mel_scale"])
    assert_close(fb.numpy(), librosa_melfb[f"fb_{i:02d}"], rtol=1.3e-6, atol=7e-5)


def test_melscale_fbanks_warning_and_errors():
    # reference functional_impl.py:1332-1349
    with pytest.warns(UserWarning, match="At least one mel filterbank has all zero values"):
        F.melscale_fbanks(201, 0.0, 8000.0, 128, 16000)
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        F.melscale_fbanks(201, 0.0, 8000.0, 64, 16000)
    with pytest.raises(ValueError):
        F.melscale_fbanks(201, 0.0, 8000.0, 64, 16000, norm="other")
    with pytest.raises(ValueError):
        F.melscale_fbanks(201, 0.0, 8000.0, 64, 16000, mel_scale="other")
    with pytest.raises(ValueError):
        F.create_dct(13, 40, "other")


def test_create_dct_norm_relation():
    # reference transforms_test.py:157-173: ortho = none * sqrt(1/(2 n_mels)), row 0 * sqrt(1/(4 n_mels))
    n_mfcc, n_mels = 40, 128
    none = F.create_dct(n_mfcc, n_mels, None)
    ortho = F.create_dct(n_mfcc, n_mels, "ortho")
    assert torch.allclose(ortho[:, 0], none[:, 0] * math.sqrt(1 / (4 * n_mels)), atol=1e-6)
    assert torch.allclose(ortho[:, 1:], none[:, 1:] * math.sqrt(1 / (2 * n_mels)), atol=1e-6)


def test_resample_kernel_dtype_rules():
    # transforms_test_impl.py:74-82 (cache dtype) + the float64-built/float32-stored default
    k32, w = F._get_sinc_resample_kernel(16000, 8000, 8000)
    assert k32.dtype == torch.float32 and w == math.ceil(6 * 2 / 0.99)
    k64, _ = F._get_sinc_resample_kernel(16000, 8000, 8000, dtype=torch.float64)
    assert k64.dtype == torch.float64
    with pytest.raises(ValueError):
        F._get_sinc_resample_kernel(16000, 8000, 8000, resampling_method="foo")
    with pytest.raises(ValueError):
        F._get_sinc_resample_kernel(16000, 8000, 8000, lowpass_filter_width=0)
    with pytest.raises(Exception, match="integer type"):
        F._get_sinc_resample_kernel(16000.5, 8000, 1)
    with pytest.warns(UserWarning, match="deprecated"):
        F._get_sinc_resample_kernel(16000, 8000, 8000, resampling_method="kaiser_window")


# ---------------- integer bookkeeping: Python and C twins vs the reference ----------------------
def test_frames_and_lengths_bit_exact(lib, ref_integers):
    for L, n_fft, hop, center, pad, t in ref_integers["stft_frames"]:
        L, n_fft, hop, center, pad, t = map(int, (L, n_fft, hop, center, pad, t))
        assert bk.num_frames(L, n_fft, hop, bool(center), pad) == t, (L, n_fft, hop, center, pad)
        assert lib.b200a_num_frames(L, n_fft, hop, center, pad) == t
    for o, n, L, w, taps, out_len in ref_integers["resample"]:
        o_r, n_r, g = bk.resample_ratio(int(o), int(n))
        assert bk.resample_width(o_r, n_r, 6, 0.99) == w == lib.b200a_resample_width(o_r, n_r, 6, 0.99)
        assert 2 * w + o_r == taps
        assert bk.resample_len(int(L), o_r, n_r) == out_len == lib.b200a_resample_len(int(L), o_r, n_r)


def test_pad_index_matches_torch_pad(lib):
    n, h = 11, 4
    x = torch.arange(n, dtype=torch.float32)[None, None]
    for mode_name, mode in _lib.PAD_MODE.items():
        ref = torch.nn.functional.pad(x + 1, (h, h), mode=mode_name)[0, 0]  # +1 so zero == padding
        for i in range(-h, n + h):
            j_c = lib.b200a_pad_index(i, n, mode)
            j_py = bk.pad_index(i, n, mode)
            assert j_c == j_py
            assert ref[i + h].item() == (0.0 if j_c < 0 else float(j_c + 1)), (mode_name, i)


def test_shard_bounds_partition():
    for total in (0, 1, 7, 256, 2048, 2049):
        for world in (1, 2, 3, 8):
            spans = [bk.shard_bounds(total, world, r) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == total
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [e - b for b, e in spans]
            assert max(sizes) - min(sizes) <= 1


# ---------------- the C ABI library ---------------------------------------------------------------
def test_library_exports_every_declared_symbol(lib):
    header = open(os.path.join(ROOT, "include", "b200audio.h")).read()
    declared = set(re.findall(r"^(?:int|size_t|int64_t|int32_t|const char\*)\s+(b200a_[a-z0-9_]+)\(", header, re.M))
    assert declared, "no declarations parsed"
    raw = ctypes.CDLL(_lib.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(raw, name), f"{name} declared in include/b200audio.h but not exported"
    assert declared == set(_lib.EXPORTED_SYMBOLS), "ctypes table and header disagree"
    assert lib.b200a_version() == 100
    assert ctypes.sizeof(_lib.FrontendDesc) == 16 * 4


def test_abi_argument_validation_without_gpu(lib):
    d = _lib.FrontendDesc()
    assert lib.b200a_frontend_workspace_bytes(d) == 0  # all-zero descriptor is invalid
    good = T.Spectrogram(n_fft=512)._frontend_plan().desc
    assert lib.b200a_frontend_workspace_bytes(good) > 512 * 4 + 512 * 8
    # null pointers / bad sizes are rejected before any CUDA call
    assert lib.b200a_frontend_run(good, None, 1, None, 1, 1000, 1000, None, None, 1, None) == _lib.EINVAL
    assert lib.b200a_frontend_prepare(good, None, None, None, None, 0, None) == _lib.EINVAL
    assert lib.b200a_resample_run(None, None, 441, 160, 17, None, 1, 10, 10, None, 10, 4, None) == _lib.EINVAL
    assert lib.b200a_fill_f32(None, 4, 0.0, None) == _lib.EINVAL
    bad = T.Spectrogram(n_fft=512)._frontend_plan().desc
    bad.hop = 0
    assert lib.b200a_frontend_workspace_bytes(bad) == 0
    big = T.Spectrogram(n_fft=16384)._frontend_plan().desc
    assert lib.b200a_frontend_workspace_bytes(big) == 0  # > 8192 is documented as unsupported
    for code in (0, -1, -2, -3, -4, -5, -99):
        assert isinstance(lib.b200a_strerror(code), bytes)
    assert lib.b200a_num_bins(1024, 1) == 513 and lib.b200a_num_bins(1024, 0) == 1024


# ---------------- drop-in module surface ----------------------------------------------------------
def test_state_dict_names_match_reference():
    # transforms_test.py:68-85
    m = T.MelSpectrogram()
    assert set(m.state_dict()) == {"spectrogram.window", "mel_scale.fb"}
    mf = T.MFCC()
    assert set(mf.state_dict()) == {"MelSpectrogram.spectrogram.window", "MelSpectrogram.mel_scale.fb", "dct_mat"}
    assert set(T.Resample(16000, 8000).state_dict()) == {"kernel"}
    assert set(T.Resample(16000, 16000).state_dict()) == set()
    assert set(T.Spectrogram().state_dict()) == {"window"}
    assert set(T.MelScale().state_dict()) == {"fb"}


def test_defaults_and_attributes():
    s = T.Spectrogram()
    assert (s.n_fft, s.win_length, s.hop_length, s.pad, s.power, s.normalized) == (400, 400, 200, 0, 2.0, False)
    assert (s.center, s.pad_mode, s.onesided) == (True, "reflect", True)
    m = T.MelSpectrogram()
    assert (m.sample_rate, m.n_fft, m.n_mels, m.f_min, m.f_max, m.hop_length) == (16000, 400, 128, 0.0, None, 200)
    assert m.mel_scale.f_max == 8000.0 and tuple(m.mel_scale.fb.shape) == (201, 128)
    mf = T.MFCC()
    assert (mf.n_mfcc, mf.dct_type, mf.norm, mf.top_db, mf.log_mels) == (40, 2, "ortho", 80.0, False)
    assert mf.amplitude_to_DB.multiplier == 10.0 and mf.amplitude_to_DB.db_multiplier == 0.0
    r = T.Resample(44100, 16000)
    assert (r.orig_freq, r.new_freq, r.gcd, r.lowpass_filter_width, r.rolloff) == (44100, 16000, 100, 6, 0.99)
    a = T.AmplitudeToDB("magnitude", 80.0)
    assert a.multiplier == 20.0 and a.amin == 1e-10 and a.ref_value == 1.0


def test_constructor_errors_match_reference():
    with pytest.raises(ValueError, match="DCT type not supported"):
        T.MFCC(dct_type=3)
    with pytest.raises(ValueError, match="Cannot select more MFCC coefficients"):
        T.MFCC(n_mfcc=60, melkwargs=dict(n_mels=40))
    with pytest.raises(ValueError, match="top_db must be positive"):
        T.AmplitudeToDB(top_db=-1.0)
    with pytest.raises(ValueError, match="Require f_min"):
        T.MelScale(f_min=9000.0, f_max=100.0)
    with pytest.raises(ValueError, match="Invalid resampling method"):
        T.Resample(16000, 8000, resampling_method="foo")
    with pytest.raises(ValueError, match="Invalid normalized parameter"):
        F._get_spec_norms("energy")
    with pytest.raises(TypeError):
        F._get_spec_norms(1.0)
    with pytest.warns(UserWarning, match="onesided"):
        T.MelSpectrogram(onesided=True)
    with pytest.warns(UserWarning, match="return_complex"):
        T.Spectrogram(return_complex=True)


def test_no_cpu_fallback():
    x = torch.randn(2, 4000)
    for mod in (T.Spectrogram(), T.MelSpectrogram(), T.MFCC(), T.Resample(16000, 8000), T.AmplitudeToDB()):
        with pytest.raises(RuntimeError, match="no CPU or ATen fallback"):
            mod(x)
    with pytest.raises(RuntimeError, match="no CPU or ATen fallback"):
        F.resample(x, 16000, 8000)
    with pytest.raises(ValueError):
        F.resample(x, 0, 8000)
    assert F.resample(x, 8000, 8000) is x  # identity fast path (functional.py:1471-1472)
    assert T.Resample(8000, 8000)(x) is x
    with pytest.raises(TypeError, match="Expected floating point type"):
        F.resample(torch.zeros(4, dtype=torch.int32), 16000, 8000)


def test_library_path_is_in_tree():
    assert audio_b200.library_path().startswith(ROOT)


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU arm the driver runs next to ours) prints ONE JSON line with the contract's
    keys; it needs no GPU, so its shape is checked here."""
    import json
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    proc = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                          capture_output=True, text=True, timeout=600, cwd=root)
    assert proc.returncode == 0, proc.stderr[-2000:]
    lines = [ln for ln in proc.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    rec = json.loads(lines[0])
    assert rec["impl"] == "reference"
    if "unavailable" in rec:
        return
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in rec, key
    assert rec["metric"] == "MelSpectrogram frames/sec" and rec["unit"] == "frames/s" and rec["value"] > 0
    assert rec["cpu_baseline"]["kind"] in ("reference", "port") and rec["cpu_baseline"]["cores"] >= 1
    assert rec["e2e"]["h2d_bytes_per_step"] == 0 and rec["e2e"]["d2h_bytes_per_step"] == 0


def test_reference_switch_routes_modules_to_torchaudio():
    """B200A_REFERENCE=1 (read at import) runs the reference class behind the same surface, loudly (warning)."""
    import subprocess
    import sys

    pytest.importorskip("torchaudio")
    code = r"""
import sys, warnings
sys.path.insert(0, sys.argv[1])
import torch
with warnings.catch_warnings(record=True) as w:
    warnings.simplefilter("always")
    import audio_b200.transforms as T
assert any("B200A_REFERENCE" in str(x.message) for x in w), "the switch must announce itself"
import torchaudio.transforms as R
x = torch.randn(2, 4000, generator=torch.Generator().manual_seed(0))
m = T.MelSpectrogram(16000, n_fft=400, hop_length=160, n_mels=40)
assert torch.equal(m(x), R.MelSpectrogram(16000, n_fft=400, hop_length=160, n_mels=40)(x))   # CPU input: reference path
m.spectrogram.window.mul_(0.5)  # the module's own buffers are what the reference run uses
assert torch.allclose(m(x), 0.25 * R.MelSpectrogram(16000, n_fft=400, hop_length=160, n_mels=40)(x), rtol=1e-5)
r = T.Resample(44100, 16000)
assert torch.equal(r(x), R.Resample(44100, 16000)(x))
print("ok")
"""
    env = dict(os.environ, B200A_REFERENCE="1")
    out = subprocess.run([sys.executable, "-c", code, ROOT], env=env, capture_output=True, text=True)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]


def test_bench_clock_sampler_pause_and_fallback():
    """bench.py's clock sampler: one per job, pausable (no query in flight inside the launch-bound e2e section), and a
    summary that says where the numbers came from.  Without a GPU both NVML and nvidia-smi are absent: the sampler must
    still start, pause, resume and stop cleanly."""
    import importlib.util
    import time

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    assert bench.E2E_WINDOWS >= 3 and bench.E2E_WINDOWS % 2 == 1  # a median needs an odd count
    with bench.ClockSampler([0], active=True, period=0.005) as c:
        time.sleep(0.03)
        c.pause()
        n = len(c.rows)
        time.sleep(0.03)
        assert len(c.rows) == n  # nothing is sampled while paused
        c.resume()
    s = c.summary()
    assert set(s) >= {"sm_mhz", "sm_max_mhz", "reasons", "source"}
    with bench.ClockSampler(range(8), active=False) as idle:  # ranks other than 0
        idle.pause()
        idle.resume()
    assert idle.rows == [] and not idle._t.is_alive()
    # both arms describe the workload with the same words (the driver pairs their lines)
    assert bench.workload_config(8)["global_batch"] == 8 * bench.BATCH


def test_bench_dump_outputs_and_steps(tmp_path):
    """`bench.py --dump-outputs`: float32 host arrays, the whole tensor when it fits, otherwise the same seeded rows on
    every run (so two builds can be compared array for array), and a hard cap on what it writes; `--steps` below 1 is
    refused instead of timing nothing."""
    import importlib.util
    import subprocess
    import sys

    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    t = torch.arange(1024 * 3, dtype=torch.float64).reshape(1024, 3)
    full = bench.dump_array(t)
    assert full.dtype == np.float32 and np.array_equal(full, t.numpy())
    a, b = bench.dump_array(t, 6 * 3 * 4), bench.dump_array(t, 6 * 3 * 4)
    assert a.dtype == np.float32 and a.shape == (6, 3) and np.array_equal(a, b)
    rows = a[:, 0] / 3
    assert np.all(np.diff(rows) > 0) and np.array_equal(a, t.numpy()[rows.astype(int)])
    assert bench.dump_array(t[:, None, :], 1).shape == (1, 1, 3)  # never less than one whole row
    bench.write_dumps(str(tmp_path / "d"), {"x": a})
    assert np.array_equal(np.load(tmp_path / "d" / "x.npy"), a)
    with pytest.raises(AssertionError, match="--dump-outputs"):
        bench.write_dumps(str(tmp_path / "big"), {"x": np.zeros(bench.DUMP_BYTES // 4 + 1, np.float32)})
    assert not (tmp_path / "big").exists()
    proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True)
    assert proc.returncode == 2 and "--steps" in proc.stderr


@pytest.mark.parametrize("method", ["sinc_interp_hann", "sinc_interp_kaiser"])
def test_resample_tc_band_covers_the_reference_kernels_support(method):
    """The tcgen05 resampler's banded plan is computed on the host from (orig', new', width) alone and assumes that
    phase j has live taps only inside (j orig'/new', j orig'/new' + 2 width).  Check that against the taps the
    reference's own construction (functional.py:1359-1400, rebuilt bit-identically in _constants) really produces, with
    the device's liveness rule (|k| > 1e-12 max|k| of the row) -- if the band were too narrow the device-side check would
    silently send every call to the slower kernel."""
    import ctypes

    from audio_b200 import _constants as C
    from audio_b200 import _lib

    L = _lib.lib()
    first, last = ctypes.c_int32(), ctypes.c_int32()
    info = (ctypes.c_int32 * 4)()
    for orig, new in [(44100, 16000), (48000, 16000), (16000, 8000), (22050, 16000), (44100, 48000), (8000, 16000),
                      (16000, 44100), (11025, 8000), (32000, 44100), (10, 11), (11, 10)]:
        g = math.gcd(orig, new)
        k, width = C.sinc_resample_kernel(orig, new, g, resampling_method=method)
        k = k[:, 0, :].double().numpy()
        o, n = orig // g, new // g
        assert k.shape == (n, 2 * width + o)
        assert L.b200a_resample_plan_info(o, n, width, info) == 0 and info[0] in (1, 2, 3)
        if info[0] == 1:
            assert o % 2 == 1 and 0 < info[1] <= 64 * 1024 and info[2] <= 227 * 1024
        for j in range(n):
            assert L.b200a_resample_tc_band(o, n, width, j, ctypes.byref(first), ctypes.byref(last)) == 0
            live = np.nonzero(np.abs(k[j]) > 1e-12 * np.abs(k[j]).max())[0]
            assert first.value <= live.min() and live.max() <= last.value, (orig, new, j, first.value, last.value)
            assert last.value - first.value <= 2 * width + 2  # and it is tight: at most two taps wider than 2 width
    assert L.b200a_resample_plan_info(441, 160, 17, info) == 0 and info[0] == 1 and info[3] == 61  # config 3
    assert L.b200a_resample_plan_info(2, 1, 13, info) == 0 and info[0] == 2  # even orig': the mma.sync kernel
    assert L.b200a_resample_plan_info(0, 1, 13, info) != 0
