"""GPU tests of the host-side product paths around the kernels: HostPipeline (the `e2e` path of bench.py), the plan
caches, the sharded MFCC with its NCCL all-reduce(MAX) (BASELINE config 4), and all-row oracle comparisons at the
benchmarked sizes."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
from conftest import scaled_tol_close

import audio_b200.functional as F
import audio_b200.transforms as T
from audio_b200.pipeline import HostPipeline
from oracle import frontend_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def randn(*shape, seed=0):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed))


# ---------------- HostPipeline ---------------------------------------------------------------------------------
@pytest.mark.parametrize("rows,chunk", [(70, 32), (64, 64), (5, 64), (129, 64), (1, 1)])
def test_host_pipeline_equals_resident(rows, chunk):
    m = T.MelSpectrogram(16000, n_fft=1024, hop_length=256, n_mels=80).to(DEV)
    x = randn(rows, 24000, seed=rows)
    pipe = HostPipeline(m, chunk_rows=chunk)
    got = pipe(x.pin_memory())
    pipe.synchronize()
    ref = m(x.to(DEV))
    assert got.shape == ref.shape and tuple(got.stride()) == (got.shape[1] * got.shape[2], 1, got.shape[1])
    assert torch.equal(got, ref.cpu())  # chunking never changes a row's arithmetic


def test_host_pipeline_back_to_back_calls_and_caller_buffer():
    m = T.MelSpectrogram(16000, n_fft=512, hop_length=128, n_mels=40).to(DEV)
    pipe = HostPipeline(m, chunk_rows=16)
    xs = [randn(50, 16000, seed=s).pin_memory() for s in range(4)]
    outs = [torch.empty((50, 126, 40)).pin_memory() for _ in range(4)]
    views = [pipe(x, o) for x, o in zip(xs, outs)]  # four calls in flight, no synchronisation in between
    pipe.join()
    torch.cuda.current_stream().synchronize()
    for x, v, o in zip(xs, views, outs):
        assert v.data_ptr() == o.data_ptr()
        assert torch.equal(v, m(x.to(DEV)).cpu())
    # a different batch shape re-allocates the staging buffers
    x2 = randn(7, 8000, seed=9)
    got = pipe(x2)
    pipe.synchronize()
    assert torch.equal(got, m(x2.to(DEV)).cpu())


def test_host_pipeline_refuses_batch_coupled_modules():
    kw = dict(n_fft=400, hop_length=160, n_mels=40)
    with pytest.raises(ValueError, match="top_db"):
        HostPipeline(T.MFCC(16000, n_mfcc=13, melkwargs=kw).to(DEV))
    with pytest.raises(ValueError, match="top_db"):
        HostPipeline(T.LFCC(16000, n_lfcc=13, speckwargs=dict(n_fft=400, hop_length=160)).to(DEV))
    mfl = T.MFCC(16000, n_mfcc=13, log_mels=True, melkwargs=kw).to(DEV)  # no clamp: rows independent
    x = randn(9, 8000, seed=3)
    pipe = HostPipeline(mfl, chunk_rows=4)
    got = pipe(x)
    pipe.synchronize()
    assert torch.equal(got, mfl(x.to(DEV)).cpu())
    with pytest.raises(TypeError):
        pipe(x.to(DEV))


# ---------------- plan caches must not confuse recycled allocations (ADVICE r1, high) ---------------------------
def test_functional_plan_cache_survives_recycled_window_address():
    x = randn(2, 8000, seed=1).to(DEV)
    args = dict(pad=0, n_fft=400, hop_length=100, win_length=400, power=2.0, normalized=False)
    ptrs = []
    for fn in (torch.hann_window, torch.hamming_window, torch.blackman_window, torch.hann_window):
        w = fn(400, device=DEV)  # a temporary: freed after the call, its address is handed to the next window
        ptrs.append(w.data_ptr())
        got = F.spectrogram(x, window=w, **args)
        exp = O.spectrogram(x.cpu().numpy(), 0, w.cpu().numpy().astype(np.float64), 400, 100, 400, 2.0)
        scaled_tol_close(got.cpu().numpy(), exp, what=fn.__name__)
        del w, got
    # (the caching allocator normally recycles the block; the assertion above is what matters either way)
    k1 = torch.ones(160 * 475, device=DEV)
    del k1


def test_resample_plan_holds_its_kernel():
    r = T.Resample(44100, 16000).to(DEV)
    x = randn(2, 9000, seed=2).to(DEV)
    y0 = r(x).clone()
    r.kernel.mul_(2.0)  # in-place edit bumps the version: the workspace must be rebuilt
    assert torch.allclose(r(x), 2.0 * y0, rtol=1e-6, atol=1e-7)


# ---------------- sharded MFCC: NCCL all-reduce(MAX) of the batch-global top_db maximum -------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _mfcc_rank(rank, world, port, path):
    import torch.distributed as dist

    sys.path.insert(0, ROOT)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world, device_id=dev)
    g = torch.Generator().manual_seed(2024)
    x = torch.randn(24, 40000, generator=g)
    x[5] *= 1e-4  # quiet rows: the clamp at (global max - 80 dB) floors them
    x[17] *= 1e-3
    mf = T.MFCC(16000, n_mfcc=40, melkwargs=dict(n_fft=1024, hop_length=256, n_mels=80)).to(dev)
    full = mf(x.to(dev))  # single-GPU answer on the whole 2-D batch
    per = 24 // world
    mf.process_group = dist.group.WORLD
    part = mf(x[rank * per:(rank + 1) * per].to(dev))
    parts = [torch.empty_like(part) for _ in range(world)]
    dist.all_gather(parts, part.contiguous())
    ok = torch.equal(torch.cat(parts, 0), full.contiguous())
    mf.process_group = None
    local = mf(x[rank * per:(rank + 1) * per].to(dev))  # without the exchange the quiet rows' shard differs
    differs = not torch.equal(local, part)
    flags = torch.tensor([int(ok), int(differs)], device=dev)
    dist.all_reduce(flags, op=dist.ReduceOp.SUM)
    if rank == 0:
        with open(path, "w") as fh:
            fh.write(f"{int(flags[0])} {int(flags[1])}")
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs (NCCL between two ranks)")
def test_sharded_mfcc_matches_single_gpu_over_nccl(tmp_path):
    import torch.multiprocessing as mp

    world = 2
    path = str(tmp_path / "result.txt")
    mp.spawn(_mfcc_rank, args=(world, _free_port(), path), nprocs=world, join=True)
    ok, differs = map(int, open(path).read().split())
    assert ok == world, "sharded MFCC + all-reduce(MAX) must reproduce the single-GPU 2-D batch bit for bit"
    assert differs >= 1, "the test batch must actually exercise the clamp (some shard changes without the exchange)"


def test_group_max_exchange_is_the_function_the_cpu_test_covers():
    # same code path as tests/test_distributed_cpu.py, here on a CUDA tensor without a group: identity
    g = torch.tensor([1.0, -3.0], device=DEV)
    assert F._exchange_group_max(g, None) is g


# ---------------- all rows against the fp64 oracle at the benchmarked sizes (VERDICT r1, weak #1) --------------------
def _all_rows(got, oracle_rows, rows, step=32, what=""):
    for lo in range(0, rows, step):
        exp = oracle_rows(lo, min(rows, lo + step))
        scaled_tol_close(got[lo:lo + step].float().cpu().numpy(), exp, what=f"{what} rows {lo}..{lo + step}")


def test_config2_every_row_against_oracle():
    B, L = 256, 160000
    x = torch.randn(B, L, device=DEV, generator=torch.Generator(device=DEV).manual_seed(1234))
    m = T.MelSpectrogram(16000, n_fft=1024, hop_length=256, n_mels=80).to(DEV)
    y = m(x)
    fb = m.mel_scale.fb.cpu().numpy()
    xh = x.cpu().numpy()
    _all_rows(y, lambda lo, hi: O.mel_spectrogram(xh[lo:hi], sample_rate=16000, n_fft=1024, hop_length=256, n_mels=80, fb=fb),
              B, what="config 2")


def test_config4_every_row_against_oracle_2d_and_3d():
    B, L = 256, 160000
    x = torch.randn(B, L, device=DEV, generator=torch.Generator(device=DEV).manual_seed(99))
    x[3] *= 1e-4
    x[200] *= 1e-5
    mf = T.MFCC(16000, n_mfcc=40, melkwargs=dict(n_fft=1024, hop_length=256, n_mels=80)).to(DEV)
    fb, dct = mf.MelSpectrogram.mel_scale.fb.cpu().numpy(), mf.dct_mat.cpu().numpy()
    kw = dict(n_fft=1024, hop_length=256, n_mels=80)
    xh = x.cpu().numpy()
    y3 = mf(x[:, None, :])[:, 0]  # per-item clamp: rows independent, chunk the oracle freely
    _all_rows(y3, lambda lo, hi: O.mfcc(xh[lo:hi, None], 16000, 40, "ortho", False, kw, fb=fb, dct=dct)[:, 0], B,
              what="config 4 (3-D)")
    # 2-D batch: ONE cut-off for all 256 rows.  The oracle needs the global maximum, so build the dB features row
    # chunk by row chunk, take the maximum over everything, then clamp + DCT.
    y2 = mf(x)
    feats = [10.0 * np.log10(np.maximum(O.mel_spectrogram(xh[lo:lo + 32], sample_rate=16000, fb=fb, **kw), 1e-10))
             for lo in range(0, B, 32)]  # (32, n_mels, T) dB, amplitude_to_DB with ref = 1 (functional.py:390-393)
    gmax = max(float(f.max()) for f in feats)
    for i, f in enumerate(feats):
        clamped = np.maximum(f, gmax - 80.0)  # :395-399 with ONE maximum over the 2-D batch
        exp = np.swapaxes(np.swapaxes(clamped, -1, -2) @ dct.astype(np.float64), -1, -2)
        scaled_tol_close(y2[32 * i:32 * i + 32].cpu().numpy(), exp, what=f"config 4 (2-D) rows {32 * i}")
    assert not torch.allclose(y2[3], y3[3])  # the quiet rows are where the two clamps differ


def test_config3_many_rows_against_oracle_and_mma_kernel():
    """At 44.1 -> 16 kHz the tcgen05 resampler walks the 32-frame tiles of several rows through one CTA: compare 256
    full-length rows with the oracle (not just the first two)."""
    B, L = 256, 220500
    x = torch.randn(B, L, device=DEV, generator=torch.Generator(device=DEV).manual_seed(4321))
    r = T.Resample(44100, 16000, resampling_method="sinc_interp_kaiser").to(DEV)
    y = r(x)
    xh = x.cpu().numpy()
    for lo in range(0, B, 32):
        exp = O.resample(xh[lo:lo + 32], 44100, 16000, resampling_method="sinc_interp_kaiser")
        err = np.abs(y[lo:lo + 32].cpu().numpy() - exp).max()
        assert err <= 1e-4 * np.abs(exp).max(), (lo, err)
