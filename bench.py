#!/usr/bin/env python
"""bench.py -- MelSpectrogram frames/s on BASELINE.json config 2, at 1..8 B200, plus every other BASELINE config.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the fused front end over one batch of synthetic waveforms:
MelSpectrogram(16 kHz, n_fft=1024, hop=256, n_mels=80) on (256, 160000) fp32 PER GPU
(weak scaling: the batch is sharded, every rank holds 256 utterances resident in HBM; no
collective is on this path).  Prints ONE JSON line on rank 0.

  value     whole-job frames/s, inputs resident in HBM (CUDA events, max over ranks)
  e2e       same metric through the public host-buffer API (audio_b200.pipeline.HostPipeline): pinned-host ->
            device copy of every step's batch and device -> host read of the result inside the timed region
  roofline  algorithmic HBM bytes per launch / kernel time vs the measured copy bandwidth
  configs   the other BASELINE configs, same timing method, each with its own roofline fraction:
            C3 Resample 44.1->16 kHz kaiser on 1024 x 220500 (out-samples/s), C4 MFCC n_mfcc=40 on a 2-D batch of
            256 x 160000 per GPU (batch-global top_db: at N > 1 the NCCL all-reduce(MAX) of the running maximum
            is INSIDE the timed region), C5 fused STFT+mel sweep n_fft in {256, 512, 1024, 2048} (hop = n_fft/4)
  cpu_baseline  the reference's CPU path (installed torchaudio wheel, hot-path source identical to
            /root/reference) or, if that cannot be imported, the numpy oracle port -- rank 0, N = 1 only
  --impl reference   the same reference CPU path as its own arm: the FULL 256 x 160000 batch per step
  --dump-outputs DIR  after the timing, rank 0 writes what the LAST timed step of each GPU section returned, as float32
            DIR/<name>.npy: the headline MelSpectrogram in full, and of the other configs a fixed seeded sample of whole
            rows (at most DUMP_SIDE_BYTES each); the e2e result is asserted equal to the headline's.  Inputs come from
            seeded generators, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
import warnings

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SAMPLE_RATE, N_FFT, HOP, N_MELS, N_MFCC = 16000, 1024, 256, 80, 40
BATCH, LENGTH = 256, 160000
FRAMES = 1 + LENGTH // HOP  # 626
RS_ROWS, RS_LEN, RS_ORIG, RS_NEW = 1024, 220500, 44100, 16000
RS_OUT = 80000
E2E_WINDOWS = 5
WORKLOAD = "MelSpectrogram n_fft=1024 hop=256 n_mels=80, batch=256x16kHzx10s fp32 per GPU (BASELINE configs[1])"
# SURVEY.md 8(d): compulsory traffic of the fused op = waveform in + features out + constant tables
ALGO_BYTES = 4 * (BATCH * LENGTH + BATCH * FRAMES * N_MELS) + 4 * (N_FFT + (N_FFT // 2 + 1) * N_MELS)
# dram__bytes_read.sum + dram__bytes_write.sum of one launch of the fused kernel (ncu --set full capture):
# the write-back of part of the 51 MB output is still in L2 at kernel end
NCU_DRAM_BYTES = 196_650_752
NCU_DRAM_SOURCE = "ncu --set full, profiles/r2_mel_v3_tc2_prefetch.txt (dram read 163.99 MB + write 32.66 MB per launch)"
DUMP_BYTES = 64 << 20  # --dump-outputs: every array together (the headline alone is 51.3 MB)
DUMP_SIDE_BYTES = 2 << 20  # --dump-outputs: each array of the other configs


def workload_config(world):
    """`config` of the JSON line -- identical for the b200 and the reference arm."""
    return {"workload": WORKLOAD, "global_batch": world * BATCH, "frames_per_step": world * BATCH * FRAMES,
            "parallelism": f"batch shard x{world}, no collective",
            "l2": "input 163.8 MB per step > 126 MB L2 (no flush needed)"}


def dump_array(t, max_bytes=None):
    """`t` as a contiguous float32 host array; above `max_bytes`, only the whole rows (dim 0) of a fixed seeded choice
    that fit, in ascending order, so every run of the same arguments samples the same rows."""
    import numpy as np
    import torch

    rows = t.shape[0]
    keep = rows if max_bytes is None else max(1, min(rows, max_bytes // (4 * t[0].numel())))
    if keep < rows:
        idx = np.sort(np.random.default_rng(0).choice(rows, keep, replace=False))
        t = t[torch.from_numpy(idx).to(t.device)]
    return np.ascontiguousarray(t.float().cpu().numpy())


def write_dumps(out_dir, arrays):
    import numpy as np

    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_BYTES, f"--dump-outputs would write {total} bytes (limit {DUMP_BYTES})"
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clocks and throttle reasons (the fields of `nvidia-smi --query-gpu=clocks.sm,clocks.max.sm,
    clocks_event_reasons.*`) sampled while the GPU sections of the bench run.

    Read through NVML inside this process (pynvml = nvidia_ml_py, the library nvidia-smi itself sits on); the nvidia-smi
    BINARY (a driver attach per sample) is only the fallback when NVML cannot be imported.  ONE sampler per job
    (rank 0) covers every GPU of the job, and it is PAUSED inside the launch-bound end-to-end section (sampled right
    before and right after it): the e2e number of the same code moved between 3.04 ms (twice), 3.9, 12.4 and 32.8 ms
    per step from box to box at N = 1 and was 6.75 ms at N = 8 with a sampler in every rank, against 4.35 ms in
    tools/h2d_probe.py, which has no sampler.  The cause was not isolated inside the round's GPU budget; keeping
    driver queries out of that 60 ms window removes the one suspect this file controls."""

    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, indices, active=True, period=0.02):
        self.rows, self._stop, self.indices, self.active = [], threading.Event(), list(indices), active
        self.period, self.source, self._nvml, self._handles = period, None, None, []
        self._paused, self._lock = threading.Event(), threading.Lock()
        self._t = threading.Thread(target=self._run, daemon=True)

    def pause(self):
        """No query is in flight or will start until resume(): the launch-bound end-to-end section is bracketed by
        samples, not interleaved with them (a driver query next to 12 CUDA API calls per 3 ms step is measurable)."""
        self._paused.set()
        with self._lock:
            pass

    def resume(self):
        self._paused.clear()

    def _open_nvml(self):
        try:
            import pynvml
            import torch

            pynvml.nvmlInit()
            for i in self.indices:
                p = torch.cuda.get_device_properties(i)
                bdf = f"{p.pci_domain_id:08x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
                try:
                    self._handles.append(pynvml.nvmlDeviceGetHandleByPciBusId(bdf.encode()))
                except Exception:
                    self._handles.append(pynvml.nvmlDeviceGetHandleByIndex(i))
            self._nvml, self.source = pynvml, "NVML (pynvml) in-process"
        except Exception:
            self._nvml, self._handles, self.source = None, [], "nvidia-smi subprocess"

    def _sample_nvml(self):
        n = self._nvml
        masks = [n.nvmlClocksEventReasonHwSlowdown, n.nvmlClocksEventReasonHwThermalSlowdown,
                 n.nvmlClocksEventReasonSwThermalSlowdown, n.nvmlClocksEventReasonSwPowerCap]
        for h in self._handles:
            sm = n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM)
            mx = n.nvmlDeviceGetMaxClockInfo(h, n.NVML_CLOCK_SM)
            reasons = n.nvmlDeviceGetCurrentClocksEventReasons(h)
            self.rows.append([str(sm), str(mx)] + ["Active" if reasons & m else "Not Active" for m in masks])

    def _sample_smi(self):
        out = subprocess.run(
            ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-i",
             ",".join(str(i) for i in self.indices)], capture_output=True, text=True, timeout=5).stdout.strip()
        for line in out.splitlines():
            if line.strip():
                self.rows.append([c.strip() for c in line.split(",")])

    def _run(self):
        while not self._stop.is_set():
            if self._paused.is_set():
                self._stop.wait(0.002)
                continue
            with self._lock:
                try:
                    if self._nvml is not None:
                        self._sample_nvml()
                    else:
                        self._sample_smi()
                except Exception:
                    pass
            self._stop.wait(self.period if self._nvml is not None else max(self.period, 0.5))

    def __enter__(self):
        if self.active:
            self._open_nvml()
            self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self.active:
            self._t.join(timeout=6)

    def summary(self):
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock query unavailable"], "source": self.source}
        reasons = set()
        for r in self.rows:
            for n, v in zip(self.NAMES, r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]), "samples": len(sm),
                "reasons": sorted(reasons), "gpus": len(self.indices), "source": self.source,
                "window": "headline timed region and configs sections; the e2e section is bracketed (sampler paused inside)"}


# ---- the reference on the host ---------------------------------------------------------------------------------
def _reference_module(kind, **kw):
    """(callable(x) running the reference's CPU path, kind, description)."""
    try:
        import torchaudio  # the image's wheel: functional.py byte-identical to /root/reference's

        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            if kind == "mel":
                mod = torchaudio.transforms.MelSpectrogram(SAMPLE_RATE, n_fft=kw["n_fft"], hop_length=kw["hop"], n_mels=N_MELS)
            elif kind == "mfcc":
                mod = torchaudio.transforms.MFCC(SAMPLE_RATE, n_mfcc=N_MFCC,
                                                 melkwargs=dict(n_fft=N_FFT, hop_length=HOP, n_mels=N_MELS))
            else:
                mod = torchaudio.transforms.Resample(RS_ORIG, RS_NEW, resampling_method="sinc_interp_kaiser")
        return (lambda x: mod(x)), "reference", f"torchaudio {torchaudio.__version__} CPU"
    except Exception as exc:  # noqa: BLE001
        from oracle import frontend_oracle as O

        if kind == "mel":
            fn = lambda x: O.mel_spectrogram(x.numpy(), sample_rate=SAMPLE_RATE, n_fft=kw["n_fft"], hop_length=kw["hop"], n_mels=N_MELS)  # noqa: E731
        elif kind == "mfcc":
            fn = lambda x: O.mfcc(x.numpy(), SAMPLE_RATE, N_MFCC, "ortho", False, dict(n_fft=N_FFT, hop_length=HOP, n_mels=N_MELS))  # noqa: E731
        else:
            fn = lambda x: O.resample(x.numpy(), RS_ORIG, RS_NEW, resampling_method="sinc_interp_kaiser")  # noqa: E731
        return fn, "port", f"numpy float64 oracle port (torchaudio not importable: {type(exc).__name__})"


def pick_threads(fn, x):
    """The reference gets the thread count it runs fastest with (all cores is often NOT the fastest for these
    small ATen ops on a 100+ core host); the count used is reported as `cores`."""
    import torch

    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    best_n, best_t = avail, float("inf")
    with torch.inference_mode():
        for n in sorted({avail, 64, 32, 16, 8}):
            if n > avail:
                continue
            torch.set_num_threads(n)
            fn(x)
            t0 = time.perf_counter()
            fn(x)
            dt = time.perf_counter() - t0
            if dt < best_t:
                best_n, best_t = n, dt
    torch.set_num_threads(best_n)
    return best_n


def time_cpu(kind, rows, length, units_per_row, unit, steps, warmup, threads=None, **kw):
    import torch

    fn, impl, desc = _reference_module(kind, **kw)
    x = torch.randn(rows, length, generator=torch.Generator().manual_seed(1234))
    cores = pick_threads(fn, x) if threads is None else threads
    torch.set_num_threads(cores)
    with torch.inference_mode():
        for _ in range(warmup):
            fn(x)
        best, total = float("inf"), 0.0
        for _ in range(steps):
            t0 = time.perf_counter()
            fn(x)
            dt = time.perf_counter() - t0
            best, total = min(best, dt), total + dt
    units = rows * units_per_row
    return {"value": units / (total / steps), "best": units / best, "unit": unit, "cores": cores, "kind": impl,
            "sample": f"{desc}; {rows}x{length} fp32 per step, mean of {steps} steps after {warmup} warm-up"}, total / steps


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    base, sec = time_cpu("mel", BATCH, LENGTH, FRAMES, "frames/s", steps=max(args.steps, 1), warmup=max(args.warmup, 1),
                         n_fft=N_FFT, hop=HOP)
    line = {
        "impl": "reference", "metric": "MelSpectrogram frames/sec", "value": base["value"], "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.gpus),
        "note": "host CPU path; every step is the full 256x160000 batch of ONE GPU's shard (the host is not "
                "replicated per GPU: frames/s does not grow with --gpus)",
        "cpu_baseline": base,
        "e2e": {"value": base["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---- the B200 arm ------------------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist

    import audio_b200.transforms as T
    from audio_b200 import _lib, _numa

    _lib.lib()  # fail loudly if the CUDA extension is missing
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run --nproc-per-node {args.gpus}")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # pinned staging buffers must be first-touched on the GPU's own NUMA node (8 ranks pulling 164 MB per step
    # across the socket link was the end-to-end scaling limiter of round 1)
    affinity0 = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
    numa = _numa.bind_to_gpu(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    K, W = args.steps, max(args.warmup, 3)

    def time_steps(fn, steps=K, warm=W):
        """(ms per step, what the last step returned): `warm` untimed steps, then `steps` steps between two CUDA events,
        barrier + sync on both sides."""
        for _ in range(warm):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps - 1):
            fn()
        out = fn()  # outside the loop: keeping every output there would hold it alive across the next step
        e1.record()
        barrier()
        return e0.elapsed_time(e1) / steps, out

    dumps = {}

    def keep(name, out, max_bytes=DUMP_SIDE_BYTES):
        if args.dump_outputs and rank == 0:
            dumps[name] = dump_array(out, max_bytes)

    def max_over_ranks(values):
        t = torch.tensor(values, device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.tolist()

    peak, peak_src = measured_peaks()
    mel = T.MelSpectrogram(SAMPLE_RATE, n_fft=N_FFT, hop_length=HOP, n_mels=N_MELS).to(dev)
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    x = torch.randn(BATCH, LENGTH, device=dev, generator=g)  # this rank's shard, resident in HBM
    configs = []

    # rank 0 samples the clocks of every GPU of the job (local ranks 0 .. world - 1 on this one node)
    with torch.inference_mode(), ClockSampler([local] if world == 1 else range(world), active=(rank == 0)) as clocks:
        # ---- headline: config 2, inputs resident -------------------------------------------------------------
        ms_step, y = time_steps(lambda: mel(x))
        keep("melspectrogram", y, max_bytes=None)

        # ---- end to end: pinned host -> device, fused kernel, device -> pinned host ----------------------------
        from audio_b200.pipeline import HostPipeline

        xh = torch.empty((BATCH, LENGTH), dtype=torch.float32).pin_memory()
        xh.copy_(x)
        yh = torch.empty((BATCH, FRAMES, N_MELS), dtype=torch.float32).pin_memory()
        pipe = HostPipeline(mel, chunk_rows=64)

        def e2e_step():
            pipe(xh, yh)

        for _ in range(2):
            e2e_step()
        pipe.join()
        clocks.pause()  # sampled right before and right after this 60 ms section, not during it
        # E2E_WINDOWS windows of exactly K steps each, every one bracketed like the headline (barrier + sync on both sides,
        # CUDA events, max over ranks); the MEDIAN window is reported and all of them are listed: a K-step window is only
        # ~60 ms of launch-bound host work, and one stall of the host (another tenant, a driver query) multiplies it
        e2e_windows = []
        for _ in range(E2E_WINDOWS):
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(K):
                e2e_step()
            pipe.join()  # the current stream waits for the last device -> host copy
            e1.record()
            barrier()
            e2e_windows.append(e0.elapsed_time(e1) / K)
        e2e_windows = max_over_ranks(e2e_windows)
        ms_e2e = sorted(e2e_windows)[len(e2e_windows) // 2]
        clocks.resume()
        # the pipelined result is the same tensor the resident path produces
        assert torch.equal(yh.to(dev).transpose(-1, -2), y), "host pipeline result differs from resident result"
        del xh, yh, pipe

        # ---- C4: MFCC on a 2-D batch (batch-global top_db); at N > 1 the all-reduce(MAX) is live ------------------
        mf = T.MFCC(SAMPLE_RATE, n_mfcc=N_MFCC, melkwargs=dict(n_fft=N_FFT, hop_length=HOP, n_mels=N_MELS)).to(dev)
        if world > 1:
            mf.process_group = dist.group.WORLD
        ms_c4, c4_out = time_steps(lambda: mf(x))
        keep("mfcc", c4_out)
        del c4_out
        mf_local = T.MFCC(SAMPLE_RATE, n_mfcc=N_MFCC, melkwargs=dict(n_fft=N_FFT, hop_length=HOP, n_mels=N_MELS)).to(dev)
        ms_c4_local = time_steps(lambda: mf_local(x))[0] if world > 1 else ms_c4
        c4_bytes = 4 * (BATCH * LENGTH + BATCH * FRAMES * N_MFCC) + 4 * (N_FFT + 513 * N_MELS + N_MELS * N_MFCC)
        del mf, mf_local

        # ---- C5: fused STFT+mel sweep, hop = n_fft / 4, batch 256 per GPU ---------------------------------------------
        sweep = []
        for n_fft in (256, 512, 1024, 2048):
            hop = n_fft // 4
            fr = 1 + LENGTH // hop
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")  # n_fft = 256 leaves two of the 80 mel filters empty (reference warns too)
                m5 = T.MelSpectrogram(SAMPLE_RATE, n_fft=n_fft, hop_length=hop, n_mels=N_MELS).to(dev)
            if n_fft == N_FFT:
                ms5 = ms_step  # the headline, dumped above
            else:
                ms5, out5 = time_steps(lambda: m5(x))
                keep(f"melspectrogram_nfft{n_fft}", out5)
                del out5
            sweep.append((n_fft, hop, fr, ms5, 4 * (BATCH * LENGTH + BATCH * fr * N_MELS) + 4 * (n_fft + (n_fft // 2 + 1) * N_MELS)))
            del m5
        del x, y
        torch.cuda.empty_cache()

        # ---- C3: Resample 44.1 -> 16 kHz, 1024 x 220500 per GPU ------------------------------------------------------
        rs = T.Resample(RS_ORIG, RS_NEW, resampling_method="sinc_interp_kaiser").to(dev)
        xr = torch.randn(RS_ROWS, RS_LEN, device=dev, generator=g)
        ms_c3, c3_out = time_steps(lambda: rs(xr))
        keep("resample", c3_out)
        c3_bytes = 4 * (RS_ROWS * RS_LEN + RS_ROWS * RS_OUT) + 4 * 160 * 475
        del xr, rs, c3_out
        torch.cuda.empty_cache()
    clock_summary = clocks.summary()
    if dumps:
        write_dumps(args.dump_outputs, dumps)

    vals = [ms_step, ms_e2e, ms_c4, ms_c4_local, ms_c3] + [s[3] for s in sweep]
    vals = max_over_ranks(vals)
    ms_step, ms_e2e, ms_c4, ms_c4_local, ms_c3 = vals[:5]
    sweep = [(s[0], s[1], s[2], v, s[4]) for s, v in zip(sweep, vals[5:])]

    if rank == 0:
        def roof(nbytes, ms):
            a = nbytes / (ms * 1e-3) / 1e9
            return {"bound": "hbm", "achieved": a, "peak": peak, "unit": "GB/s", "frac": a / peak, "algorithmic_bytes": nbytes}

        frames_job = world * BATCH * FRAMES
        configs.append({"key": "C3", "name": "C3 Resample 44.1kHz->16kHz sinc_interp_kaiser, 1024x220500 fp32 per GPU",
                        "metric": "output samples/sec", "unit": "out-samples/s", "ms_per_step": ms_c3,
                        "value": world * RS_ROWS * RS_OUT / (ms_c3 * 1e-3), "roofline": roof(c3_bytes, ms_c3)})
        configs.append({"key": "C4", "name": "C4 MFCC n_mfcc=40 (MelSpec+dB+DCT), 2-D batch 256x160000 per GPU, batch-global top_db"
                                + (f"; all-reduce(MAX) over {world} ranks (NCCL) inside the step" if world > 1 else ""),
                        "metric": "MFCC frames/sec", "unit": "frames/s", "ms_per_step": ms_c4,
                        "value": frames_job / (ms_c4 * 1e-3), "roofline": roof(c4_bytes, ms_c4),
                        "ms_per_step_without_collective": ms_c4_local,
                        "collective_cost_ms": ms_c4 - ms_c4_local if world > 1 else 0.0})
        for n_fft, hop, fr, ms5, nbytes in sweep:
            configs.append({"key": f"C5 n_fft={n_fft}", "name": f"C5 MelSpectrogram n_fft={n_fft} hop={hop} n_mels=80, 256x160000 per GPU",
                            "metric": "MelSpectrogram frames/sec", "unit": "frames/s", "ms_per_step": ms5,
                            "value": world * BATCH * fr / (ms5 * 1e-3), "roofline": roof(nbytes, ms5)})
        line = {
            "metric": "MelSpectrogram frames/sec", "value": frames_job / (ms_step * 1e-3), "unit": "frames/s",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(world),
            "roofline": dict(roof(ALGO_BYTES, ms_step), traffic=NCU_DRAM_BYTES, traffic_source=NCU_DRAM_SOURCE,
                             peak_source=peak_src, kernel="fused STFT+mel kernel (one launch per step)"),
            "e2e": {"value": frames_job / (ms_e2e * 1e-3), "unit": "frames/s",
                    "h2d_bytes_per_step": BATCH * LENGTH * 4, "d2h_bytes_per_step": BATCH * FRAMES * N_MELS * 4,
                    "ms_per_step": ms_e2e, "windows_ms_per_step": [round(w, 4) for w in e2e_windows],
                    "estimator": f"median of {E2E_WINDOWS} windows of {K} steps",
                    "api": "audio_b200.pipeline.HostPipeline(chunk_rows=64)",
                    "numa": numa},
            "gpu_launches": K,
            "clocks": clock_summary,
            "configs": configs,
        }
        if world == 1:
            if affinity0 is not None:
                os.sched_setaffinity(0, affinity0)  # the CPU reference gets every host core back
            base, _ = time_cpu("mel", BATCH, LENGTH, FRAMES, "frames/s", steps=5, warmup=1, n_fft=N_FFT, hop=HOP)
            line["cpu_baseline"] = base
            th = base["cores"]
            cpu = {}
            cpu["C3"], _ = time_cpu("resample", 64, RS_LEN, RS_OUT, "out-samples/s", steps=2, warmup=1, threads=th)
            cpu["C4"], _ = time_cpu("mfcc", 32, LENGTH, FRAMES, "frames/s", steps=2, warmup=1, threads=th)
            for n_fft in (256, 512, 2048):
                cpu[f"C5 n_fft={n_fft}"], _ = time_cpu("mel", 32, LENGTH, 1 + LENGTH // (n_fft // 4), "frames/s", steps=2,
                                                       warmup=1, threads=th, n_fft=n_fft, hop=n_fft // 4)
            cpu["C5 n_fft=1024"] = base
            for c in configs:
                if c["key"] in cpu:
                    c["cpu_baseline"] = cpu[c["key"]]
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of each GPU section returned to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the GPU sections; the reference arm has none")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
