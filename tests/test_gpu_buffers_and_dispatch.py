"""Every kernel launch path at its dispatch boundaries, through the C ABI with caller-owned guarded buffers.

The header promises that the caller owns every buffer and that plain float pointers may sit at any 4-byte offset
(complex64 ones at any 8-byte offset).  Each operand here lives inside a larger device buffer filled with a quiet-NaN
sentinel, at float offset 0..3, with a row pitch larger than the row where the entry point takes a stride, and with
4 KiB of sentinel before and after.  After each call:
  (i)   guards, pitch gaps and columns the call does not own still hold the sentinel, bit for bit;
  (ii)  no sentinel is left anywhere in the logical output (nothing was skipped);
  (iii) the output is bit-identical with the same call on fresh, aligned, contiguous buffers;
and the result is compared with the fp64 oracle.  A sample read from outside an input view is a NaN and turns the
outputs it reaches into NaN, even where a zero tap or window weight multiplies it.

The boundaries of the dispatch matrix are computed from the formulas the launchers use (constants cited next to
them), and both sides of each are run.  The resampler's kernel family is also asserted on the host alone
(b200a_resample_plan_info), so that a change of launch logic that moves a cell to another family fails without a GPU.
"""
import ctypes
import math
import re
import warnings

import numpy as np
import pytest
import torch
from conftest import assert_close, scaled_tol_close

import audio_b200.functional as F
import audio_b200.transforms as T
from audio_b200 import _build, _lib
from audio_b200._plans import FrontendPlan, ResamplePlan
from oracle import frontend_oracle as O

DEV = "cuda:0"
SENTINEL = 0x7FC0DEAD  # a quiet NaN with a payload no arithmetic produces
GUARD = 1024  # floats of sentinel before and after each operand: 4 KiB
gpu = pytest.mark.gpu


def _stream():
    return torch.cuda.current_stream().cuda_stream


# ---------------------------------------------------------------------------------------------------------------------
# guarded buffers
# ---------------------------------------------------------------------------------------------------------------------
class Guarded:
    """`rows` x `width` floats placed `offset` floats into a sentinel-filled device buffer, rows `pitch` floats apart."""

    def __init__(self, rows, width, pitch=None, offset=0, data=None):
        self.rows, self.width = rows, width
        self.pitch = width if pitch is None else pitch
        self.start = GUARD + offset
        self.n = rows * self.pitch
        self.bits = torch.full((2 * GUARD + offset + self.n,), SENTINEL, dtype=torch.int32, device=DEV)
        self.view = self._grid(self.bits.view(torch.float32))[:, :width]
        self.owned = torch.zeros(self.bits.shape, dtype=torch.bool, device=DEV)
        self._grid(self.owned)[:, :width] = True
        if data is not None:
            self.view.copy_(torch.as_tensor(data, dtype=torch.float32).reshape(rows, width))

    def _grid(self, t):
        return t[self.start : self.start + self.n].view(self.rows, self.pitch)

    def disown(self, cols):
        """Columns of each row the call must leave alone."""
        self._grid(self.owned)[:, cols] = False

    @property
    def ptr(self):
        return self.bits.data_ptr() + 4 * self.start

    def check(self, what, written=True):
        """(i) and, for outputs, (ii)."""
        torch.cuda.synchronize()
        bits = self.bits.cpu().numpy()
        owned = self.owned.cpu().numpy()
        bad = np.flatnonzero((bits != SENTINEL) & ~owned)
        assert bad.size == 0, (f"{what}: {bad.size} floats outside the operand were written, first at buffer float "
                               f"{bad[0]} (operand starts at {self.start}, pitch {self.pitch}, width {self.width})")
        if written:
            miss = np.flatnonzero((bits == SENTINEL) & owned)
            assert miss.size == 0, f"{what}: {miss.size} output floats never written, first at buffer float {miss[0]}"

    def values(self):
        return self.view.cpu().numpy()


def bits_equal(a, b, what):
    a = a.contiguous().view(torch.int32).cpu()
    b = b.contiguous().view(torch.int32).cpu()
    assert a.shape == b.shape, f"{what}: shape {tuple(a.shape)} vs {tuple(b.shape)}"
    diff = (a != b).nonzero()
    assert diff.shape[0] == 0, f"{what}: {diff.shape[0]} floats differ from the fresh-buffer call, first at {diff[0].tolist()}"


def ok(rc, where):
    assert rc == _lib.OK, f"{where}: status {rc} ({_lib.lib().b200a_strerror(rc).decode()})"


def randn(*shape, seed):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed))


# ---------------------------------------------------------------------------------------------------------------------
# front end: one cell = one descriptor and stage, run guarded and fresh, compared with the fp64 oracle
# ---------------------------------------------------------------------------------------------------------------------
def stage_limit_hop(n_fft):
    """Largest hop for which a unit of the register-FFT kernel fits its staging buffer (frontend_pow2.cu, frontend_run_pow2:
    stage_ok = n_fft + (frames_per_unit - 1) * hop <= stage_floats); above it edge units take the 64-bit gather."""
    G = n_fft // 32
    frames_per_unit = 2 * (32 // G)
    stage_floats = 2 * (32 // G) * (32 * (G + 1) + (8 if G == 8 else 0))
    return (stage_floats - n_fft) // (frames_per_unit - 1)


def mel_fb(n_fft, n_mels, kind="htk", sample_rate=16000):
    n_freqs = n_fft // 2 + 1
    if kind == "dense":  # every bin feeds every filter: no band structure
        return torch.rand(n_freqs, n_mels, generator=torch.Generator().manual_seed(n_fft + n_mels))
    f_min, f_max, norm, scale = 0.0, float(sample_rate // 2), None, "htk"
    if kind == "narrow":
        f_min, f_max = 4000.0, 8000.0
    elif kind == "slaney":
        norm, scale = "slaney", "slaney"
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")  # empty filters at small n_fft
        return F.melscale_fbanks(n_freqs, f_min, f_max, n_mels, sample_rate, norm, scale)


def frontend_cell(n_fft, hop, stage, power=2.0, fb=None, log_mels=False, rows=3, length=None, in_off=1, in_pad=5,
                  out_off=3, gmax_rows_per_group=None, seed=0):
    """Run one b200a_frontend_run call guarded and fresh; return (frame-major output, group maxima or None, oracle)."""
    lib = _lib.lib()
    n_mels = 0 if fb is None else fb.shape[1]
    if length is None:
        length = 12 * hop + n_fft + 37
    desc = FrontendPlan.make_desc(n_fft, n_fft, hop, 0, True, "reflect", True, False, False,
                                  None if stage == _lib.STAGE_COMPLEX else power, n_mels=n_mels, log_mels=log_mels)
    plan = FrontendPlan(desc)
    window = torch.hann_window(n_fft)
    ws = plan.workspace(window.to(DEV), None if fb is None else fb.to(DEV), None)
    frames = plan.frames(length)
    n_bins = n_fft // 2 + 1
    width = n_mels if stage >= _lib.STAGE_MEL else n_bins
    per_frame = 2 * width if stage == _lib.STAGE_COMPLEX else width
    x = randn(rows, length, seed=seed + n_fft + hop)
    rpg = gmax_rows_per_group or rows
    groups = -(-rows // rpg)
    if stage == _lib.STAGE_COMPLEX:
        out_off &= ~1  # complex64 output: 8-byte aligned (4-byte aligned is EINVAL, see the test below)

    def call(wave_ptr, row_stride, out_ptr, gmax_ptr):
        ok(lib.b200a_frontend_run(desc, ws.data_ptr(), stage, wave_ptr, rows, length, row_stride, out_ptr, gmax_ptr, rpg,
                                  _stream()), f"frontend_run n_fft={n_fft} hop={hop} stage={stage}")

    g_in = Guarded(rows, length, pitch=length + in_pad, offset=in_off, data=x)
    g_out = Guarded(rows * frames, per_frame, offset=out_off)
    g_max = None
    if stage == _lib.STAGE_FEAT and gmax_rows_per_group is not None:
        g_max = Guarded(1, groups, offset=(out_off + 1) % 4, data=torch.full((groups,), -math.inf))
    call(g_in.ptr, length + in_pad, g_out.ptr, None if g_max is None else g_max.ptr)
    what = f"n_fft={n_fft} hop={hop} stage={stage} power={power} n_mels={n_mels}"
    g_in.check(what + " (input)", written=False)
    g_out.check(what)

    xd = x.to(DEV)
    fresh = torch.empty(rows * frames, per_frame, device=DEV)
    fresh_max = torch.full((groups,), -math.inf, device=DEV) if g_max is not None else None
    call(xd.data_ptr(), length, fresh.data_ptr(), None if fresh_max is None else fresh_max.data_ptr())
    bits_equal(g_out.view, fresh, what)
    if g_max is not None:
        g_max.check(what + " (group_max)")
        bits_equal(g_max.view.reshape(-1), fresh_max, what + " (group_max)")

    got = g_out.values().reshape(rows, frames, per_frame)
    spec = O.spectrogram(x.numpy(), 0, window.numpy(), n_fft, hop, n_fft, None if stage == _lib.STAGE_COMPLEX else power)
    exp = np.swapaxes(spec, -1, -2)  # frame-major
    if stage == _lib.STAGE_COMPLEX:
        got = got[..., 0::2] + 1j * got[..., 1::2]
    elif stage >= _lib.STAGE_MEL:
        exp = exp @ fb.double().numpy()
    return got, (None if g_max is None else g_max.values().reshape(-1)), exp


def check_frontend(got, exp, stage, log_mels, what):
    if stage != _lib.STAGE_FEAT:
        scaled_tol_close(got, exp, what=what)
        return
    # dB / log features: back to the mel domain, where the 1e-4 rule of the other stages applies
    if log_mels:
        scaled_tol_close(np.exp(got.astype(np.float64)) - 1e-6, exp, what=what)
    else:
        scaled_tol_close(10.0 ** (got.astype(np.float64) / 10.0), np.maximum(exp, 1e-10), what=what)


STAGES = {"complex": _lib.STAGE_COMPLEX, "power": _lib.STAGE_POWER, "mel": _lib.STAGE_MEL}


def _staging_hops():
    cells = []
    for n_fft in (256, 512, 1024):
        lim = stage_limit_hop(n_fft)
        for hop in sorted({lim, lim + 1, n_fft, n_fft + n_fft // 3 + 1}):
            cells.append((n_fft, hop))
    # n_fft 2048 runs on its own kernels (stft2048_*); hops across eo_frame_bulk_ok's range and beyond n_fft
    cells += [(2048, 512), (2048, 1089), (2048, 2048), (2048, 2731)]
    return cells


def test_staging_limit_formula():
    """The hops the staging cells straddle (they are derived, not copied: this pins the derivation)."""
    assert [stage_limit_hop(n) for n in (256, 512, 1024)] == [301, 554, 1088]


@gpu
@pytest.mark.parametrize("stage", sorted(STAGES))
@pytest.mark.parametrize("n_fft,hop", _staging_hops())
def test_frontend_staging_limit(n_fft, hop, stage):
    st = STAGES[stage]
    fb = mel_fb(n_fft, 40) if st == _lib.STAGE_MEL else None
    got, _, exp = frontend_cell(n_fft, hop, st, fb=fb)
    check_frontend(got, exp, st, False, f"n_fft={n_fft} hop={hop} {stage}")


HG8_STAGES = [("complex", _lib.STAGE_COMPLEX, False), ("power", _lib.STAGE_POWER, False), ("mel", _lib.STAGE_MEL, False),
              ("feat_db", _lib.STAGE_FEAT, False), ("feat_log", _lib.STAGE_FEAT, True)]


@gpu
@pytest.mark.parametrize("power", [2.0, 1.0, 0.5, 3.0])
@pytest.mark.parametrize("name,stage,log_mels", HG8_STAGES, ids=[s[0] for s in HG8_STAGES])
def test_frontend_hg8_specialisation(name, stage, log_mels, power):
    """n_fft 1024, hop 256 and a 16-byte aligned input with a pitch of a multiple of 4 take the HG=8 kernels
    (launch_g: bulk_ok && hop == 256); the same signal at float offset 1 takes HG=-1.  Same bits either way."""
    if stage == _lib.STAGE_COMPLEX and power != 2.0:
        pytest.skip("the complex stage has no power")
    fb = mel_fb(1024, 80) if stage >= _lib.STAGE_MEL else None
    rpg = 2 if stage == _lib.STAGE_FEAT else None
    # length and pitch multiples of 4: the aligned call (and the fresh one inside frontend_cell) stage in bulk
    kw = dict(fb=fb, power=power, log_mels=log_mels, rows=4, gmax_rows_per_group=rpg, length=40 * 256 + 516)
    got8, max8, exp = frontend_cell(1024, 256, stage, in_off=0, in_pad=4, out_off=0, **kw)
    got1, max1, _ = frontend_cell(1024, 256, stage, in_off=1, in_pad=4, out_off=2, **kw)
    assert np.array_equal(got8, got1), "HG=8 and HG=-1 differ"
    check_frontend(got8, exp, stage, log_mels, f"{name} power={power}")
    if max8 is not None:
        assert np.array_equal(max8, max1)
        if not log_mels:
            db = 10.0 * np.log10(np.maximum(exp, 1e-10))
            exp_max = db.reshape(2, -1).max(axis=1)  # rows_per_group = 2 of 4 rows
            assert_close(max8, exp_max, rtol=1e-4, atol=1e-3, what="group_max")


MEL_BODY_CELLS = [(n_fft, n_mels) for n_fft in (256, 512, 1024) for n_mels in (1, 8, 127, 128, 129, 511, 512, 513)]


def test_mel_body_boundaries():
    """128 filters is the tcgen05 limit (kTcMaxN), 512 the contraction plan's (kMaxItems groups of 8 filters)."""
    kTcMaxN, kMaxItems = 128, 64
    n_mels = sorted({m for _, m in MEL_BODY_CELLS})
    for lim in (kTcMaxN, 8 * kMaxItems):
        assert {lim - 1, lim, lim + 1} <= set(n_mels)


@gpu
@pytest.mark.parametrize("n_fft,n_mels", MEL_BODY_CELLS)
def test_mel_contraction_bodies(n_fft, n_mels):
    fb = mel_fb(n_fft, n_mels)
    got, _, exp = frontend_cell(n_fft, n_fft // 4, _lib.STAGE_MEL, fb=fb, length=20 * n_fft + 11)
    scaled_tol_close(got, exp, what=f"n_fft={n_fft} n_mels={n_mels}")


FB_CELLS = [(2048, 128, "htk"), (2048, 512, "htk"), (2048, 128, "dense"), (2048, 512, "dense"), (1024, 128, "dense"),
            (1024, 128, "narrow"), (1024, 80, "slaney"), (2048, 128, "narrow"), (2048, 128, "slaney"), (512, 64, "narrow")]


@gpu
@pytest.mark.parametrize("n_fft,n_mels,kind", FB_CELLS)
def test_mel_filterbank_shapes(n_fft, n_mels, kind):
    """Dense filterbanks at n_fft 2048 have more fragment steps than stay in shared memory (kEoFragSteps = 136) and
    read the rest from global memory; narrow-band and slaney banks change the band plan."""
    fb = mel_fb(n_fft, n_mels, kind)
    for stage in (_lib.STAGE_MEL, _lib.STAGE_FEAT):
        got, _, exp = frontend_cell(n_fft, n_fft // 4, stage, fb=fb, length=16 * n_fft + 3,
                                    gmax_rows_per_group=1 if stage == _lib.STAGE_FEAT else None)
        check_frontend(got, exp, stage, False, f"n_fft={n_fft} n_mels={n_mels} {kind} stage={stage}")


# ---------------------------------------------------------------------------------------------------------------------
# MFCC finish: kernel selection (frontend_generic.cu, mfcc_finish_impl)
# ---------------------------------------------------------------------------------------------------------------------
MFCC_CELLS = [  # (n_mels, n_mfcc, clamp, kernel the launcher picks)
    (128, 64, True, "mma"),        # clamp and n_mfcc <= 64, tables <= 200 KB
    (80, 40, False, "tiled5"),     # no clamp, n_mfcc <= 40
    (128, 50, False, "tiled8"),    # no clamp, 40 < n_mfcc <= 64
    (512, 64, True, "big_clamp"),  # clamp, mma tables > 200 KB: falls through
    (128, 80, True, "generic"),    # n_mfcc > 64
    (128, 80, False, "generic"),
    (36, 13, False, "tiled5"),     # n_mels % 4 == 0: the float4 feature load, when `feat` is aligned
    (23, 13, True, "mma"),         # n_mels % 4 != 0: scalar loads
]


def mfcc_kernel_choice(n_mels, n_mfcc, clamp):
    """mfcc_finish_impl's selection, restated: shared memory of the mma / tiled kernels against the 200 KB they may use."""
    if n_mfcc <= 64 and clamp:
        ksteps, ntiles = -(-n_mels // 8), -(-n_mfcc // 8)
        if 16 * ksteps * ntiles * 32 + 4 * (128 * (8 * ksteps + 4) + 128) <= 200 * 1024:
            return "mma"
    if n_mfcc <= 64:
        cpt = 5 if n_mfcc <= 40 else 8
        if 4 * (n_mels * 8 * cpt + 128 * (n_mels + 2)) <= 200 * 1024:
            return f"tiled{cpt}"
    return "generic"


def test_mfcc_finish_cells_cover_every_kernel():
    picks = {mfcc_kernel_choice(m, c, cl) for m, c, cl, _ in MFCC_CELLS}
    assert picks == {"mma", "tiled5", "tiled8", "generic"}
    for m, c, cl, name in MFCC_CELLS:
        if name != "big_clamp":
            assert mfcc_kernel_choice(m, c, cl) == name, (m, c, cl)
        else:
            assert mfcc_kernel_choice(m, c, cl) != "mma"


@gpu
@pytest.mark.parametrize("dims", [2, 3])
@pytest.mark.parametrize("n_mels,n_mfcc,clamp,name", MFCC_CELLS)
def test_mfcc_finish_kernels(n_mels, n_mfcc, clamp, name, dims):
    """2-D input: one clamp over the batch (rows_per_group = rows); 3-D: one per item of 2 channels."""
    lib = _lib.lib()
    rows, frames = 4, 301
    rpg = rows if dims == 2 else 2
    groups = rows // rpg
    desc = FrontendPlan.make_desc(256, 256, 64, 0, True, "reflect", True, False, False, 2.0, n_mels=n_mels,
                                  n_mfcc=n_mfcc, log_mels=not clamp)
    plan = FrontendPlan(desc)
    dct = torch.as_tensor(O.create_dct(n_mfcc, n_mels, "ortho"), dtype=torch.float32)
    ws = plan.workspace(torch.hann_window(256, device=DEV), torch.zeros(129, n_mels, device=DEV), dct.to(DEV))
    g = torch.Generator().manual_seed(n_mels * 100 + n_mfcc)
    feat = torch.rand(rows * frames, n_mels, generator=g) * 120.0 - 100.0  # dB-like values
    gmax = feat.reshape(groups, -1).max(dim=1).values - torch.rand(groups, generator=g) * 5.0
    top_db = 80.0 if clamp else -1.0

    def call(feat_ptr, gmax_ptr, out_ptr):
        ok(lib.b200a_mfcc_finish(desc, ws.data_ptr(), feat_ptr, rows, frames, gmax_ptr if clamp else None, rpg, top_db,
                                 out_ptr, _stream()), f"mfcc_finish {name}")

    what = f"{name} n_mels={n_mels} n_mfcc={n_mfcc} clamp={clamp} dims={dims}"
    results = []
    for off in (1, 0, 2, 3):  # offset 1 first: a misaligned feature pointer with n_mels % 4 == 0
        g_feat = Guarded(rows * frames, n_mels, offset=off, data=feat)
        g_max = Guarded(1, groups, offset=(off + 2) % 4, data=gmax)
        g_out = Guarded(rows * frames, n_mfcc, offset=(off + 3) % 4)
        call(g_feat.ptr, g_max.ptr, g_out.ptr)
        g_feat.check(what + " (feat)", written=False)
        g_max.check(what + " (group_max)", written=False)
        g_out.check(what)
        results.append(g_out.view.clone())
    fd, md = feat.to(DEV), gmax.to(DEV)
    fresh = torch.empty(rows * frames, n_mfcc, device=DEV)
    call(fd.data_ptr(), md.data_ptr(), fresh.data_ptr())
    for r in results:
        bits_equal(r, fresh, what)
    f64 = feat.double().numpy().reshape(groups, -1, n_mels)
    if clamp:
        f64 = np.maximum(f64, gmax.double().numpy()[:, None, None] - top_db)
    exp = f64.reshape(-1, n_mels) @ dct.double().numpy()
    assert_close(results[0].cpu().numpy(), exp, rtol=1e-4, atol=5e-3, what=what)


# ---------------------------------------------------------------------------------------------------------------------
# Kaldi front end: energy column, out_col0 and columns no one owns
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("padded,n_mels", [(512, 23), (512, 80), (1024, 40)])
def test_kaldi_run_columns(padded, n_mels):
    from audio_b200.compliance import kaldi as K

    lib = _lib.lib()
    size, shift, rows, length = padded * 25 // 32, padded * 5 // 16, 3, 16000 + 7
    window = torch.zeros(padded)
    window[:size] = K._feature_window_function("povey", size, 0.42, torch.device("cpu"), torch.float32)
    bins, _ = K.get_mel_banks(n_mels, padded, 16000.0, 20.0, 0.0, 100.0, -500.0, 1.0)
    fb = torch.nn.functional.pad(bins.to(torch.float32), (0, 1)).T.contiguous()
    desc = FrontendPlan.make_desc(padded, padded, shift, 0, False, "reflect", True, False, False, 2.0, n_mels=n_mels)
    ws = FrontendPlan(desc).workspace(window.to(DEV), fb.to(DEV), None)
    for snip in (1, 0):
        kd = _lib.KaldiDesc()
        kd.window_size, kd.window_shift, kd.padded_size = size, shift, padded
        kd.snip_edges, kd.remove_dc_offset, kd.preemphasis = snip, 1, 0.97
        kd.energy_mode, kd.energy_floor, kd.use_log = 1, 0.0, 1
        # [energy | gap | n_mels values | gap]: columns 1 and out_width - 1 belong to no one
        kd.energy_col, kd.out_col0, kd.out_width = 0, 2, n_mels + 3
        frames = lib.b200a_kaldi_num_frames(length, size, shift, snip)
        x = randn(rows, length, seed=padded + n_mels + snip)

        def call(wave_ptr, row_stride, out_ptr):
            ok(lib.b200a_kaldi_run(kd, desc, ws.data_ptr(), _lib.STAGE_MEL, wave_ptr, rows, length, row_stride, out_ptr,
                                   _stream()), "kaldi_run")

        what = f"kaldi padded={padded} n_mels={n_mels} snip_edges={snip}"
        g_in = Guarded(rows, length, pitch=length + 3, offset=2, data=x)
        g_out = Guarded(rows * frames, kd.out_width, offset=1)
        g_out.disown([1, kd.out_width - 1])
        call(g_in.ptr, length + 3, g_out.ptr)
        g_in.check(what + " (input)", written=False)
        g_out.check(what)
        fresh = torch.full((rows * frames, kd.out_width), 0.0, device=DEV)
        xd = x.to(DEV)
        call(xd.data_ptr(), length, fresh.data_ptr())
        owned = [0] + list(range(2, 2 + n_mels))
        bits_equal(g_out.view[:, owned], fresh[:, owned], what)


# ---------------------------------------------------------------------------------------------------------------------
# stand-alone stages
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("off", [0, 1, 2, 3])
def test_apply_fbank_strided(off):
    lib = _lib.lib()
    rows, n_bins, frames, n_filters = 3, 257, 97, 40
    st_frame, st_bin = n_bins + 3, 1           # frame-major rows of a padded buffer
    st_row = frames * st_frame + 5
    spec = torch.rand(rows, frames, n_bins, generator=torch.Generator().manual_seed(off))
    fb = mel_fb(512, n_filters)
    # rows of `frames` frames of st_frame floats, n_bins of them data: the gaps keep the sentinel
    g_spec = Guarded(rows, frames * st_frame, pitch=st_row, offset=off)
    g_spec.view.view(rows, frames, st_frame)[:, :, :n_bins] = spec.to(DEV)
    g_fb = Guarded(n_bins, n_filters, offset=(off + 1) % 4, data=fb)
    g_out = Guarded(rows * frames, n_filters, offset=(off + 2) % 4)
    ok(lib.b200a_apply_fbank(g_spec.ptr, rows, n_bins, frames, st_row, st_bin, st_frame, g_fb.ptr, n_filters, g_out.ptr,
                             _stream()), "apply_fbank")
    g_spec.check("apply_fbank (input)", written=False)
    g_out.check("apply_fbank")
    fresh = torch.empty(rows * frames, n_filters, device=DEV)
    sd, fd = spec.to(DEV), fb.to(DEV)
    ok(lib.b200a_apply_fbank(sd.data_ptr(), rows, n_bins, frames, frames * n_bins, 1, n_bins, fd.data_ptr(), n_filters,
                             fresh.data_ptr(), _stream()), "apply_fbank")
    bits_equal(g_out.view, fresh, "apply_fbank")
    exp = spec.double().numpy() @ fb.double().numpy()
    scaled_tol_close(g_out.values().reshape(rows, frames, n_filters), exp, what="apply_fbank")


@gpu
@pytest.mark.parametrize("top_db", [80.0, -1.0])
@pytest.mark.parametrize("off", [0, 1, 3])
def test_amplitude_to_db_groups(off, top_db):
    lib = _lib.lib()
    groups, elems = 5, 3 * 1000 + 1
    x = torch.rand(groups, elems, generator=torch.Generator().manual_seed(off)) ** 8
    g_x = Guarded(groups, elems, offset=off, data=x)
    g_scratch = Guarded(1, groups, offset=(off + 1) % 4)
    g_out = Guarded(groups, elems, offset=(off + 2) % 4)
    ok(lib.b200a_amplitude_to_db(g_x.ptr, groups, elems, 10.0, 1e-10, 0.0, top_db, g_scratch.ptr, g_out.ptr, _stream()),
       "amplitude_to_db")
    g_x.check("amplitude_to_db (input)", written=False)
    g_scratch.check("amplitude_to_db (scratch)", written=top_db >= 0)
    g_out.check("amplitude_to_db")
    xd = x.to(DEV)
    fresh, scratch = torch.empty(groups, elems, device=DEV), torch.empty(groups, device=DEV)
    ok(lib.b200a_amplitude_to_db(xd.data_ptr(), groups, elems, 10.0, 1e-10, 0.0, top_db, scratch.data_ptr(),
                                 fresh.data_ptr(), _stream()), "amplitude_to_db")
    bits_equal(g_out.view, fresh, "amplitude_to_db")
    exp = 10.0 * np.log10(np.maximum(x.double().numpy(), 1e-10))
    if top_db >= 0:
        exp = np.maximum(exp, exp.max(axis=1, keepdims=True) - top_db)
    assert_close(g_out.values(), exp, rtol=1e-5, atol=1e-4, what="amplitude_to_db")


@gpu
@pytest.mark.parametrize("n_fft,hop", [(512, 128), (1024, 256), (400, 100), (256, 64)])
def test_istft_guarded(n_fft, hop):
    """istft_pow2_kernel (256 / 512 / 1024) and istft_frames_kernel (any other size); complex input at an 8-byte
    offset with padded frames, output rows at a pitch, the frame scratch guarded."""
    lib = _lib.lib()
    rows, frames = 3, 41
    bins = n_fft // 2 + 1
    desc = FrontendPlan.make_desc(n_fft, n_fft, hop, 0, True, "reflect", True, False, False, None)
    window = torch.hann_window(n_fft)
    ws = FrontendPlan(desc).workspace(window.to(DEV), None, None)
    g = torch.Generator().manual_seed(n_fft + hop)
    spec = torch.complex(torch.randn(rows, bins, frames, generator=g), torch.randn(rows, bins, frames, generator=g))
    start, out_len = n_fft // 2, hop * (frames - 1)
    s_frame = bins + 1  # complex elements; frames stored with one spare complex between them
    s_row = frames * s_frame + 3
    s_bin = 1

    def call(spec_ptr, sr, sb, sf, buf_ptr, out_ptr, out_stride):
        ok(lib.b200a_istft_run(desc, ws.data_ptr(), spec_ptr, rows, frames, sr, sb, sf, buf_ptr, out_ptr, out_stride, start,
                               out_len, _stream()), f"istft n_fft={n_fft}")

    for off in (0, 2):
        g_spec = Guarded(rows, 2 * frames * s_frame, pitch=2 * s_row, offset=off)
        grid = g_spec.view.view(rows, frames, s_frame, 2)
        grid[:, :, :bins, 0] = spec.real.transpose(1, 2).to(DEV)
        grid[:, :, :bins, 1] = spec.imag.transpose(1, 2).to(DEV)
        g_buf = Guarded(1, rows * frames * n_fft, offset=off + 1)
        g_out = Guarded(rows, out_len, pitch=out_len + 3, offset=3 - off)
        call(g_spec.ptr, s_row, s_bin, s_frame, g_buf.ptr, g_out.ptr, out_len + 3)
        g_buf.check("istft (frame scratch)", written=False)
        g_out.check(f"istft n_fft={n_fft} off={off}")
        spec_d = torch.view_as_real(spec).to(DEV).contiguous()
        buf = torch.empty(rows * frames * n_fft, device=DEV)
        fresh = torch.empty(rows, out_len, device=DEV)
        call(spec_d.data_ptr(), bins * frames, frames, 1, buf.data_ptr(), fresh.data_ptr(), out_len)
        bits_equal(g_out.view, fresh, f"istft n_fft={n_fft}")
    exp = O.istft(spec.numpy(), n_fft, hop, n_fft, window.numpy(), center=True, length=out_len)
    scaled_tol_close(g_out.values(), exp, what=f"istft n_fft={n_fft} hop={hop}")


# ---------------------------------------------------------------------------------------------------------------------
# complex pointers must be 8-byte aligned (host-side validation: nothing is launched, no device needed)
# ---------------------------------------------------------------------------------------------------------------------
FAKE = 1 << 20  # a device address is never dereferenced on the host: validation rejects the call first


@pytest.fixture(scope="module")
def clib():
    _build.build()
    return _lib.lib()


def test_complex_pointers_need_8_byte_alignment(clib):
    desc = FrontendPlan.make_desc(512, 512, 128, 0, True, "reflect", True, False, False, None)
    bad, good = FAKE + 4, FAKE
    ein = _lib.EINVAL
    assert clib.b200a_frontend_run(desc, good, _lib.STAGE_COMPLEX, good, 1, 4096, 4096, bad, None, 1, None) == ein
    assert clib.b200a_istft_run(desc, good, bad, 1, 8, 2056, 1, 257, good, good, 4096, 256, 1024, None) == ein
    for rebuilt, tprev, proj in ((bad, None, good), (good, bad, good), (good, good, bad), (None, None, bad)):
        assert clib.b200a_griffinlim_update(good, 2056, 8, 1, 0.5, rebuilt, tprev, 0.99, 1, proj, 1, 257, 8, None) == ein
    assert clib.b200a_phase_vocoder(bad, 2056, 8, 1, 1, 257, 8, 1.3, good, good, 7, None) == ein
    assert clib.b200a_phase_vocoder(good, 2056, 8, 1, 1, 257, 8, 1.3, good, bad, 7, None) == ein
    assert clib.b200a_ratio_f32(bad, 10, good, None) == ein


# ---------------------------------------------------------------------------------------------------------------------
# resampler: family per cell (host) and every cell guarded (device)
# ---------------------------------------------------------------------------------------------------------------------
TC, MMA, DIRECT = 1, 2, 3  # b200a_resample_plan_info info[0]
kTcMaxPhases, kTcMaxKSteps, kRsMaxTiles = 160, 30, 128  # resample.cu: rs_tc_steps, rs_choose
KAISER_BEST = dict(lowpass_filter_width=64, rolloff=0.9475937167399596, resampling_method="sinc_interp_kaiser",
                   beta=14.769656459379492)
KAISER_FAST = dict(lowpass_filter_width=16, rolloff=0.85, resampling_method="sinc_interp_kaiser", beta=8.555504641634386)
RS_CELLS = [  # (orig, new, kwargs, family)
    (44100, 16000, {}, TC),                             # 441:160, 475 taps = 30 k-steps: both tcgen05 limits met
    (44100, 16000, dict(lowpass_filter_width=7), MMA),  # 481 taps: 31 k-steps
    (163, 160, {}, TC),                                 # new' = 160
    (163, 161, {}, MMA),                                # new' = 161
    (22050, 16000, {}, MMA),                            # 441:320
    (44100, 16000, KAISER_BEST, MMA),
    # 147:160, 283 taps: inside both tcgen05 limits, but upsampling with a 136-tap band makes every 16-tap step touch
    # all 160 phases, and the banded blocks (18 steps x 160 phases x 64 B = 180 KiB) do not fit next to the operands
    (44100, 48000, KAISER_BEST, MMA),
    (48000, 44100, KAISER_BEST, MMA),                   # even orig'
    (44100, 16000, KAISER_FAST, MMA),
    (44100, 48000, KAISER_FAST, TC),
    (48000, 44100, KAISER_FAST, MMA),
    (48000, 44100, {}, MMA),
    (16000, 8000, {}, MMA),
    (2003, 1999, {}, DIRECT),                           # 250 phase groups of 8 > kRsMaxTiles
]
RS_IDS = [f"{o}-{n}-{kw.get('lowpass_filter_width', 6)}-{kw.get('rolloff', 0.99)}" for o, n, kw, _ in RS_CELLS]


def _ratio(orig, new, kw):
    g = math.gcd(orig, new)
    o, n = orig // g, new // g
    lpw, rolloff = kw.get("lowpass_filter_width", 6), kw.get("rolloff", 0.99)
    width = math.ceil(lpw * o / (min(o, n) * rolloff))
    return o, n, width


@pytest.mark.parametrize("orig,new,kw,family", RS_CELLS, ids=RS_IDS)
def test_resample_family_on_host(clib, orig, new, kw, family):
    o, n, width = _ratio(orig, new, kw)
    assert clib.b200a_resample_width(o, n, kw.get("lowpass_filter_width", 6), kw.get("rolloff", 0.99)) == width
    info = (ctypes.c_int32 * 4)()
    ok(clib.b200a_resample_plan_info(o, n, width, info), "resample_plan_info")
    taps = 2 * width + o
    tc_limits = o % 2 == 1 and -(-taps // 16) <= kTcMaxKSteps and n <= kTcMaxPhases
    assert family != TC or tc_limits, "the cell's family contradicts the tcgen05 limits"
    if tc_limits and family != TC:  # only the banded blocks' shared memory can rule tcgen05 out
        assert info[1] == 0 and (o, n, width) == (147, 160, 68)
    if family == DIRECT:
        assert -(-n // 8) > kRsMaxTiles
    assert info[0] == family, f"{o}:{n} width {width} ({taps} taps): family {info[0]}, expected {family}"


def test_resample_cells_straddle_the_tcgen05_limits():
    steps = {}
    for orig, new, kw, _ in RS_CELLS:
        o, n, width = _ratio(orig, new, kw)
        if o % 2:
            steps[(o, n, width)] = (-(-(2 * width + o) // 16), n)
    assert any(k == kTcMaxKSteps for k, _ in steps.values()) and any(k == kTcMaxKSteps + 1 for k, _ in steps.values())
    assert any(n == kTcMaxPhases for _, n in steps.values()) and any(n == kTcMaxPhases + 1 for _, n in steps.values())


def resample_guarded(r, x, in_off, in_pad, out_off, out_pad, what):
    """One b200a_resample_run call guarded and one fresh; returns the guarded result."""
    lib = _lib.lib()
    o, n = r.orig_freq // r.gcd, r.new_freq // r.gcd
    plan = ResamplePlan(o, n, r.width)
    ws, k = plan.workspace(r.kernel)
    rows, length = x.shape
    out_len = O.resample_len(length, o, n)

    def call(wave_ptr, row_stride, out_ptr, out_stride):
        ok(lib.b200a_resample_run(ws.data_ptr(), k.data_ptr(), o, n, r.width, wave_ptr, rows, length, row_stride, out_ptr,
                                  out_stride, out_len, _stream()), what)

    g_in = Guarded(rows, length, pitch=length + in_pad, offset=in_off, data=x)
    g_out = Guarded(rows, out_len, pitch=out_len + out_pad, offset=out_off)
    call(g_in.ptr, length + in_pad, g_out.ptr, out_len + out_pad)
    g_in.check(what + " (input)", written=False)
    g_out.check(what)
    xd = x.to(DEV)
    fresh = torch.empty(rows, out_len, device=DEV)
    call(xd.data_ptr(), length, fresh.data_ptr(), out_len)
    bits_equal(g_out.view, fresh, what)
    return g_out.values()


# (input offset, input pitch pad, output offset, output pitch pad): every output alignment mod 16 bytes, odd and even
# pitches, and an output at 4 mod 8 bytes behind an even pitch (the mma kernel's paired store must stand down)
RS_LAYOUTS = [(0, 0, 0, 0), (1, 5, 3, 2), (2, 3, 1, 3), (3, 1, 2, 4)]


@gpu
@pytest.mark.parametrize("orig,new,kw,family", RS_CELLS, ids=RS_IDS)
def test_resample_cells_guarded(orig, new, kw, family):
    o, n, width = _ratio(orig, new, kw)
    r = T.Resample(orig, new, **kw).to(DEV)
    kernel = r.kernel.cpu().double().numpy()
    # a whole number of input frames, so that the last output frame is complete (its last phase is inside out_len),
    # and a ragged length
    for length in (o * max(3, 24000 // o), o * max(3, 24000 // o) + 7):
        x = randn(3, length, seed=o + n + length)
        exp = O.apply_sinc_resample_kernel(x.numpy(), orig, new, r.gcd, kernel, width)
        for lay in RS_LAYOUTS:
            what = f"{orig}->{new} {kw} L={length} layout={lay}"
            got = resample_guarded(r, x, *lay, what)
            assert got.shape == exp.shape
            assert np.abs(got - exp).max() <= 1e-4 * np.abs(exp).max(), what


@gpu
def test_resample_device_side_fallback():
    """A live tap outside the band the tcgen05 plan assumes: the host still picks tcgen05 for 441:160, the plan kernel
    finds the tap, resample_tc_kernel leaves, and the mma.sync kernel launched behind it does the work."""
    lib = _lib.lib()
    r = T.Resample(44100, 16000).to(DEV)
    o, n, width = 441, 160, r.width
    info = (ctypes.c_int32 * 4)()
    ok(lib.b200a_resample_plan_info(o, n, width, info), "plan_info")
    assert info[0] == TC
    x = randn(2, 441 * 50, seed=11)
    r(x.to(DEV))  # builds the plan for the unedited kernel
    first, last = ctypes.c_int32(), ctypes.c_int32()
    ok(lib.b200a_resample_tc_band(o, n, width, 80, first, last), "tc_band")
    assert first.value > 10
    with torch.no_grad():
        r.kernel[80, 0, first.value - 7] = 0.25  # in place: the version stamp makes the plan rebuild
    exp = O.apply_sinc_resample_kernel(x.numpy(), 44100, 16000, r.gcd, r.kernel.cpu().double().numpy(), width)
    got = r(x.to(DEV)).cpu().numpy()
    assert np.abs(got - exp).max() <= 1e-4 * np.abs(exp).max()
    got = resample_guarded(r, x, 1, 3, 3, 2, "fallback")
    assert np.abs(got - exp).max() <= 1e-4 * np.abs(exp).max()


# ---------------------------------------------------------------------------------------------------------------------
# large indices and batch limits
# ---------------------------------------------------------------------------------------------------------------------
def need_bytes(n):
    free, _ = torch.cuda.mem_get_info()
    if free < n * 1.15:
        pytest.skip(f"needs {n / 2**30:.1f} GiB of free device memory, {free / 2**30:.1f} GiB free")


def rs_points(xrow, first, kernel, o, n, width, ms):
    """Outputs `ms` of _apply_sinc_resample_kernel for one row, from the samples xrow = x[first : first + len]
    (zero outside the row, as the reference's padding; the caller passes enough of the row)."""
    out = []
    for m in ms:
        f, j = divmod(int(m), n)
        lo = f * o - width  # x index of tap 0
        seg = np.zeros(kernel.shape[1])
        a, b = max(lo, first), min(lo + kernel.shape[1], first + len(xrow))
        if b > a:
            seg[a - lo : b - lo] = xrow[a - first : b - first]
        out.append(float(kernel[j] @ seg))
    return np.array(out)


@gpu
def test_mel_batch_over_2_31_elements():
    rows, length = 13500, 160000
    need_bytes(4 * rows * length * 1.35)
    m = T.MelSpectrogram(16000, n_fft=1024, hop_length=256, n_mels=80).to(DEV)
    x = torch.empty(rows, length, device=DEV).normal_(generator=torch.Generator(DEV).manual_seed(3))
    y = m(x)
    fb = m.mel_scale.fb.cpu().numpy()
    for r in (0, (1 << 31) // length, rows - 1):
        exp = O.mel_spectrogram(x[r : r + 1].cpu().numpy(), sample_rate=16000, n_fft=1024, hop_length=256, n_mels=80, fb=fb)
        scaled_tol_close(y[r : r + 1].cpu().numpy(), exp, what=f"row {r}")
    del x, y
    torch.cuda.empty_cache()


@gpu
def test_resample_batch_over_2_31_elements():
    rows, length = 9800, 220500
    need_bytes(4 * rows * length * 1.4)
    r = T.Resample(44100, 16000).to(DEV)
    x = torch.empty(rows, length, device=DEV).normal_(generator=torch.Generator(DEV).manual_seed(4))
    y = r(x)
    for row in (0, (1 << 31) // length, rows - 1):
        exp = O.resample(x[row].cpu().numpy(), 44100, 16000)
        got = y[row].cpu().numpy()
        assert np.abs(got - exp).max() <= 1e-4 * np.abs(exp).max(), row
    del x, y
    torch.cuda.empty_cache()


@gpu
def test_one_row_over_2_31_samples():
    """stage_ok (32-bit staged indices) and the tcgen05 length guard switch to their 64-bit paths."""
    length = (1 << 31) + 4099
    hop, n_fft = 256, 1024
    frames = 1 + length // hop
    need_bytes(4 * length + 4 * frames * 80 + 4 * (length * 16 // 44 + 4096))
    x = torch.empty(1, length, device=DEV).normal_(generator=torch.Generator(DEV).manual_seed(5))
    m = T.MelSpectrogram(16000, n_fft=n_fft, hop_length=hop, n_mels=80).to(DEV)
    y = m(x)[0]  # (80, frames)
    assert y.shape[-1] == frames
    fb = m.mel_scale.fb.cpu().numpy()
    head = x[0, : 64 * hop].cpu().numpy()
    exp = O.mel_spectrogram(head[None], sample_rate=16000, n_fft=n_fft, hop_length=hop, n_mels=80, fb=fb)[0]
    scaled_tol_close(y[:, :8].cpu().numpy(), exp[:, :8], what="first frames")
    s = (length // hop - 64) * hop  # a frame boundary: frame t of the tail is frame s/hop + t of the row
    tail = x[0, s:].cpu().numpy()
    exp = O.mel_spectrogram(tail[None], sample_rate=16000, n_fft=n_fft, hop_length=hop, n_mels=80, fb=fb)[0]
    scaled_tol_close(y[:, -8:].cpu().numpy(), exp[:, -8:], what="last frames")
    del y
    torch.cuda.empty_cache()

    r = T.Resample(44100, 16000).to(DEV)
    z = r(x)[0]
    out_len = O.resample_len(length, 441, 160)
    assert z.shape[-1] == out_len
    kernel = r.kernel.cpu().double().numpy().reshape(160, -1)
    ms = np.arange(0, 2000)
    got = z[:2000].cpu().numpy()
    exp = rs_points(x[0, :8000].cpu().numpy(), 0, kernel, 441, 160, r.width, ms)
    assert np.abs(got - exp).max() <= 1e-4 * np.abs(exp).max(), "first outputs"
    ms = np.arange(out_len - 2000, out_len)
    first = length - 8000
    exp = rs_points(x[0, first:].cpu().numpy(), first, kernel, 441, 160, r.width, ms)
    got = z[out_len - 2000 :].cpu().numpy()
    assert np.abs(got - exp).max() <= 1e-4 * max(np.abs(exp).max(), 1e-3), "last outputs"
    del x, z
    torch.cuda.empty_cache()


ROWS_64K = 65536  # one more than gridDim.y allows


def _match_or_unsupported(rc, g_out, where):
    """A batch the launcher cannot grid must be refused with EUNSUPPORTED and leave the output untouched."""
    if rc == _lib.EUNSUPPORTED:
        g_out.check(where + " (refused)", written=False)
        return False
    ok(rc, where)
    g_out.check(where)
    return True


@gpu
def test_65536_rows_resample_direct():
    lib = _lib.lib()
    r = T.Resample(2003, 1999).to(DEV)
    ws, k = ResamplePlan(2003, 1999, r.width).workspace(r.kernel)
    length = 2003 * 2
    out_len = O.resample_len(length, 2003, 1999)
    x = torch.empty(ROWS_64K, length, device=DEV).normal_(generator=torch.Generator(DEV).manual_seed(6))
    g_out = Guarded(ROWS_64K, out_len, offset=1)
    rc = lib.b200a_resample_run(ws.data_ptr(), k.data_ptr(), 2003, 1999, r.width, x.data_ptr(), ROWS_64K, length, length,
                                g_out.ptr, out_len, out_len, _stream())
    if _match_or_unsupported(rc, g_out, "resample direct"):
        for row in (0, ROWS_64K - 1):
            exp = O.resample(x[row].cpu().numpy(), 2003, 1999)
            assert np.abs(g_out.view[row].cpu().numpy() - exp).max() <= 1e-4 * np.abs(exp).max()


@gpu
def test_65536_rows_standalone_stages():
    lib = _lib.lib()
    # apply_fbank: rows on gridDim.y
    n_bins, frames, n_filters = 17, 3, 4
    spec = torch.rand(ROWS_64K, n_bins, frames, device=DEV)
    fb = torch.rand(n_bins, n_filters, device=DEV)
    g_out = Guarded(ROWS_64K * frames, n_filters)
    rc = lib.b200a_apply_fbank(spec.data_ptr(), ROWS_64K, n_bins, frames, n_bins * frames, frames, 1, fb.data_ptr(),
                               n_filters, g_out.ptr, _stream())
    if _match_or_unsupported(rc, g_out, "apply_fbank"):
        exp = spec[-1].T.double().cpu().numpy() @ fb.double().cpu().numpy()
        scaled_tol_close(g_out.values()[-frames:], exp)
    # amplitude_to_db: groups on gridDim.y
    elems = 16
    xs = torch.rand(ROWS_64K, elems, device=DEV)
    scratch = torch.empty(ROWS_64K, device=DEV)
    g_out = Guarded(ROWS_64K, elems)
    rc = lib.b200a_amplitude_to_db(xs.data_ptr(), ROWS_64K, elems, 10.0, 1e-10, 0.0, 80.0, scratch.data_ptr(), g_out.ptr,
                                   _stream())
    if _match_or_unsupported(rc, g_out, "amplitude_to_db"):
        exp = 10.0 * np.log10(np.maximum(xs[-1].double().cpu().numpy(), 1e-10))
        assert_close(g_out.values()[-1], np.maximum(exp, exp.max() - 80.0), rtol=1e-5, atol=1e-4)
    # phase vocoder: rows on gridDim.y
    bins, frames_in, rate = 9, 4, 1.5
    frames_out = math.ceil(frames_in / rate)
    spec_c = torch.randn(ROWS_64K, bins, frames_in, 2, device=DEV)
    pa = torch.linspace(0, math.pi * 4, bins, device=DEV)
    g_out = Guarded(ROWS_64K * frames_out, 2 * bins)
    rc = lib.b200a_phase_vocoder(spec_c.data_ptr(), bins * frames_in, frames_in, 1, ROWS_64K, bins, frames_in, rate,
                                 pa.data_ptr(), g_out.ptr, frames_out, _stream())
    if _match_or_unsupported(rc, g_out, "phase_vocoder"):
        sp = torch.view_as_complex(spec_c[-1]).cpu().numpy()
        exp = O.phase_vocoder(sp, rate, pa.cpu().numpy()[:, None]).T
        got = g_out.values()[-frames_out:]
        assert_close(got[:, 0::2] + 1j * got[:, 1::2], exp, rtol=1e-4, atol=1e-4)


@gpu
def test_65536_rows_istft():
    lib = _lib.lib()
    n_fft, hop, frames = 256, 64, 3
    bins = n_fft // 2 + 1
    desc = FrontendPlan.make_desc(n_fft, n_fft, hop, 0, True, "reflect", True, False, False, None)
    window = torch.hann_window(n_fft)
    ws = FrontendPlan(desc).workspace(window.to(DEV), None, None)
    spec = torch.randn(ROWS_64K, bins, frames, 2, device=DEV)
    buf = torch.empty(ROWS_64K * frames * n_fft, device=DEV)
    out_len = hop * (frames - 1)
    g_out = Guarded(ROWS_64K, out_len)
    rc = lib.b200a_istft_run(desc, ws.data_ptr(), spec.data_ptr(), ROWS_64K, frames, bins * frames, frames, 1,
                             buf.data_ptr(), g_out.ptr, out_len, n_fft // 2, out_len, _stream())
    if _match_or_unsupported(rc, g_out, "istft"):
        sp = torch.view_as_complex(spec[-1]).cpu().numpy()
        exp = O.istft(sp, n_fft, hop, n_fft, window.numpy(), center=True, length=out_len)
        scaled_tol_close(g_out.values()[-1], exp)


# ---------------------------------------------------------------------------------------------------------------------
# launch census
# ---------------------------------------------------------------------------------------------------------------------
@gpu
def test_launch_census():
    """A compact replay of the matrix under torch.profiler: every kernel family reachable with default settings runs."""
    from torch.profiler import ProfilerActivity, profile

    x = randn(2, 20000, seed=1).to(DEV)
    x_off = torch.zeros(2, 20001, device=DEV)[:, 1:]
    x_off.copy_(x)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        mods = [T.Spectrogram(n_fft=n, hop_length=n // 4).to(DEV) for n in (256, 512, 1024)]
        mods += [T.Spectrogram(n_fft=1024, hop_length=256).to(DEV), T.MelSpectrogram(16000, n_fft=512, n_mels=40).to(DEV),
                 T.Spectrogram(n_fft=2048, hop_length=512).to(DEV), T.MelSpectrogram(16000, n_fft=2048, n_mels=128).to(DEV),
                 T.Spectrogram(n_fft=400).to(DEV),
                 T.MFCC(16000, n_mfcc=40, melkwargs=dict(n_fft=512, n_mels=64)).to(DEV),
                 T.MFCC(16000, n_mfcc=13, log_mels=True, melkwargs=dict(n_fft=512, n_mels=64)).to(DEV),
                 T.MFCC(16000, n_mfcc=80, melkwargs=dict(n_fft=512, n_mels=128)).to(DEV),
                 T.Resample(44100, 16000).to(DEV), T.Resample(16000, 8000).to(DEV), T.Resample(2003, 1999).to(DEV)]
        inv = [T.InverseSpectrogram(n_fft=512).to(DEV), T.InverseSpectrogram(n_fft=400).to(DEV)]
        specs = [T.Spectrogram(n_fft=512, power=None).to(DEV)(x), T.Spectrogram(n_fft=400, power=None).to(DEV)(x)]
        for m in mods:  # plans and workspaces are built outside the profiled window
            m(x)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for m in mods:
                m(x)
            mods[2](x_off)  # n_fft 1024 / hop 256 at an unaligned address: HG = -1
            for m, s in zip(inv, specs):
                m(s)
            torch.cuda.synchronize()
    names = {e.name for e in prof.events()}
    ours = {n for n in names if "kernel" in n}
    if not ours:
        pytest.skip("the profiler returned no CUDA kernel records")
    listing = "\n".join(sorted(ours))

    def launched(pattern):
        return any(re.search(pattern, n) for n in ours)

    pow2 = [re.search(r"stft_pow2_power_kernel<[^,]+,\s*(\d+),\s*(-?\d+),", n) for n in ours]
    gs = {int(m.group(1)) for m in pow2 if m}
    hgs = {int(m.group(2)) for m in pow2 if m}
    assert gs >= {8, 16, 32}, listing
    assert hgs >= {8, -1}, listing
    for fam in ("stft_pow2_mel_kernel", "stft2048_power_kernel", "stft2048_mel_kernel", "stft_generic_kernel",
                "mfcc_finish_mma_kernel", "mfcc_finish_tiled_kernel", r"mfcc_finish_kernel\b", "resample_tc_kernel",
                "resample_mma_kernel", "resample_direct_kernel", "istft_pow2_kernel", "istft_frames_kernel"):
        assert launched(fam), f"{fam} was not launched; launched:\n{listing}"
