#!/usr/bin/env python
"""Benchmark of the chowdsp_fft hot path on B200 (DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic input.  Default workload =
BASELINE.json configs[1]: batched complex C2C N=4096 x 65536 transforms fp32, ordered, 1 GPU
(4 GiB algorithmic bytes per step; inputs + outputs are far larger than the 126 MB L2, so no L2 flush
is needed between iterations).  Prints ONE JSON line on rank 0.

  value        whole-job throughput, inputs resident in HBM, CUDA-event timed on the launch stream
  e2e          same metric through the C ABI with HOST (pinned) buffers: H2D + transform + D2H timed
  roofline     algorithmic bytes / launch duration vs the measured HBM peak (MEASURED_PEAKS.json)
  cpu_baseline the reference's own AVX build (oracle/_ref) one thread per host core, bounded sample
--impl reference runs ONLY that CPU arm (rank 0), as the driver's comparison line.

Other workloads (--workload): the remaining BASELINE configs and size variants, same JSON shape.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback
METRIC = "batched fp32 FFT throughput, algorithmic bytes (in+out) per second"


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def host_cores():
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    return n


class ClockSampler:
    """Samples SM clock / throttle reasons through NVML during the timed region."""

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self._nvml = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nvml = None

    def _run(self):
        n = self._nvml
        names = {
            n.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
            n.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            n.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            n.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            n.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(n.nvmlDeviceGetClockInfo(self._h, n.NVML_CLOCK_SM))
                r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.02)

    def __enter__(self):
        if self._nvml is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


# ======================================================================================================
# workloads
# ======================================================================================================
class BatchedFFT:
    """`batch` independent transforms of size N per GPU (weak scaling: every rank runs the same batch)."""

    scaling = "weak"

    def __init__(self, name, N, is_complex, batch, ordered, desc):
        self.name, self.N, self.is_complex, self.batch, self.ordered, self.desc = name, N, is_complex, batch, ordered, desc
        self.nfl = 2 * N if is_complex else N
        # SURVEY.md §8(d): C2C 16 N bytes per transform (8N in + 8N out); R2C 8 N bytes
        self.bytes_step = batch * (16 * N if is_complex else 8 * N)
        self.flops_step = batch * (5.0 if is_complex else 2.5) * N * math.log2(N)
        logm = int(math.log2(N)) - (0 if is_complex else 1)
        self.kernel = "cfb::fft_kernel<%d,16,%s,%d>" % (logm, "C2C_FWD" if is_complex else "R2C", 0 if ordered else 3)

    def config(self):
        return {"workload": self.desc, "N": self.N, "transform": "C2C" if self.is_complex else "R2C",
                "batch_per_gpu": self.batch, "ordered": self.ordered,
                "l2_policy": "inputs+outputs (%.1f GiB per GPU) far exceed the 126 MB L2; no flush needed" % (2 * self.batch * self.nfl * 4 / 2**30),
                "sharding": "independent transforms split by batch across GPUs, no collectives"}

    def setup(self, cf, torch, rank, world):
        self.cf, self.torch = cf, torch
        self.plan = cf.fft_new_setup(self.N, cf.FFT_COMPLEX if self.is_complex else cf.FFT_REAL, True)
        gen = torch.Generator(device="cuda").manual_seed(42 + rank)
        self.x = torch.rand(self.batch, self.nfl, device="cuda", generator=gen) * 2 - 1
        self.y = torch.empty_like(self.x)

    def step(self, stream):
        self.cf.fft_transform_batched(self.plan, self.x, self.y, self.batch, self.nfl, self.nfl, self.cf.FFT_FORWARD, self.ordered, stream)

    def outputs(self):
        """what one step hands its caller, each array as rows of its last dimension (--dump-outputs samples rows)"""
        return {"y": self.y}

    def parity(self):
        from oracle import oracle as o

        sel = self.torch.arange(0, self.batch, max(1, self.batch // 64), device="cuda")[:64]
        want = o.np_transform(self.x[sel].cpu().numpy(), self.N, self.is_complex, 8, False, self.ordered)
        return {"rel_l2_vs_oracle": o.rel_l2(self.y[sel].cpu().numpy(), want), "tolerance": o.parity_tol(self.N), "transforms": int(sel.numel())}

    def e2e(self, steps, barrier, reduce_max):
        """HOST pinned buffers through the C ABI: H2D + kernel + D2H inside the timed region."""
        cf, torch = self.cf, self.torch
        hin, hout = cf.aligned_array(self.batch * self.nfl), cf.aligned_array(self.batch * self.nfl)
        hin.reshape(self.batch, self.nfl)[:] = self.x.cpu().numpy()
        call = lambda: cf.fft_transform_batched(self.plan, hin, hout, self.batch, self.nfl, self.nfl, cf.FFT_FORWARD, self.ordered)
        call()  # warm-up (allocates the staging buffers)
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            call()
        torch.cuda.synchronize()
        dt = reduce_max((time.perf_counter() - t0) / steps)
        nchk = min(4, self.batch) * self.nfl
        ok = bool(np.array_equal(hout.reshape(-1)[:nchk], self.y.reshape(-1)[:nchk].cpu().numpy()))
        cf.aligned_free(hin.ctypes.data)
        cf.aligned_free(hout.ctypes.data)
        return {"seconds": dt, "h2d_bytes_per_step": self.batch * self.nfl * 4, "d2h_bytes_per_step": self.batch * self.nfl * 4,
                "matches_device_path": ok,
                "path": "fft_transform_batched(host pinned in/out): 32 MiB chunks, H2D/kernel/D2H overlapped on two streams"}

    def cpu(self, seconds_target, steps=1, warmup=0):
        """The unmodified reference, one thread per core over a bounded sample of the batch."""
        from oracle import oracle as o

        ref = o.load_ref()
        if ref is None:
            raise RuntimeError("oracle/_ref/libchowdsp_fft_ref.so is missing (build it with make -C oracle)")
        cores = min(ref.hardware_threads(), host_cores())
        sample = min(self.batch, max(cores * 256, 2048))
        rng = np.random.default_rng(42)
        xin = o.aligned_copy(rng.uniform(-1, 1, sample * self.nfl).astype(np.float32))
        out = o.aligned_empty(sample * self.nfl)
        run = lambda reps=1: ref.transform_timed(xin, out, self.N, self.is_complex, False, self.ordered, sample, self.nfl, self.nfl, cores, reps=reps)
        t1 = run()
        reps = max(1, int(seconds_target / max(t1, 1e-6) / max(1, steps + warmup)))
        times = [run(reps) for _ in range(warmup + steps)][warmup:]  # seconds of the threaded region only (plan / threads made outside)
        per_step = float(np.mean(times))
        gbs = sample * reps * (self.bytes_step / self.batch) / per_step / 1e9
        desc = f"{sample} transforms x {reps} passes per step, {cores} threads (one per core, pinned), reference AVX build W=32B"
        return gbs, cores, desc, per_step * 1e3


class STFT(BatchedFFT):
    """BASELINE configs[2]: R2C N=2048 hop 512 over 1024 channels x 10 s @ 48 kHz, channels sharded over GPUs."""

    scaling = "strong"

    def __init__(self):
        self.name, self.N, self.hop, self.channels_total, self.samples = "stft", 2048, 512, 1024, 480000
        self.is_complex, self.ordered, self.nfl = False, True, 2048
        self.frames = (self.samples - self.N) // self.hop + 1  # 934
        self.desc = "multichannel STFT: R2C N=2048 hop 512, 1024 channels x 480000 samples (BASELINE configs[2])"
        self.kernel = "cfb::fft_kernel<10,16,R2C,0>"

    def config(self):
        return {"workload": self.desc, "N": self.N, "hop": self.hop, "channels": self.channels_total, "frames_per_channel": self.frames,
                "transform": "R2C", "ordered": True, "window": "rectangular (the reference has none)",
                "bytes": "unique input + packed output (frames overlap 4x; re-reads hit L2)",
                "l2_policy": "9.8 GB per step across the job, far larger than L2",
                "sharding": "channels split contiguously across GPUs, no collectives"}

    def setup(self, cf, torch, rank, world):
        from chowdsp_fft_b200.sharding import shard_range

        self.cf, self.torch = cf, torch
        _, self.channels = shard_range(self.channels_total, rank, world)
        self.batch = self.channels * self.frames
        self.bytes_step = self.channels * self.samples * 4 + self.batch * self.N * 4
        self.flops_step = self.batch * 2.5 * self.N * math.log2(self.N)
        self.plan = cf.fft_new_setup(self.N, cf.FFT_REAL, True)
        gen = torch.Generator(device="cuda").manual_seed(42 + rank)
        self.x = torch.rand(self.channels, self.samples, device="cuda", generator=gen) * 2 - 1
        self.y = torch.empty(self.channels, self.frames, self.N, device="cuda")

    def step(self, stream):
        self.cf.fft_transform_strided(self.plan, self.x, self.y, self.channels, self.frames, self.samples, self.hop,
                                      self.frames * self.N, self.N, self.cf.FFT_FORWARD, True, stream)

    def parity(self):
        from oracle import oracle as o

        c = self.channels - 1
        sig = self.x[c].cpu().numpy()
        fr = np.stack([sig[f * self.hop:f * self.hop + self.N] for f in range(0, self.frames, 37)])
        got = self.y[c, ::37].cpu().numpy()
        return {"rel_l2_vs_oracle": o.rel_l2(got, o.np_transform(fr, self.N, False, 8, False, True)), "tolerance": o.parity_tol(self.N), "transforms": len(fr)}

    def e2e(self, steps, barrier, reduce_max):
        """fft_stft_forward on HOST (pinned) audio: every channel's samples cross PCIe once, spectra come back; bounded to a
        slice of the channels so that the pinned allocations stay small (the per-channel cost is what is measured)."""
        cf, torch = self.cf, self.torch
        ch = min(self.channels, 64)
        hin = cf.aligned_array(ch * self.samples).reshape(ch, self.samples)
        hout = cf.aligned_array(ch * self.frames * self.N).reshape(ch, self.frames, self.N)
        hin[:] = self.x[:ch].cpu().numpy()
        call = lambda: cf.fft_stft_forward(self.plan, hin, hout, ch, self.frames, self.samples, self.hop, self.frames * self.N, self.N, None, True)
        call()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            call()
        dt = reduce_max((time.perf_counter() - t0) / steps)
        ok = bool(np.array_equal(hout[:2], self.y[:2].cpu().numpy()))
        frac = ch / self.channels
        cf.aligned_free(hin.ctypes.data)
        cf.aligned_free(hout.ctypes.data)
        return {"seconds": dt / frac, "h2d_bytes_per_step": int(self.channels * self.samples * 4), "d2h_bytes_per_step": int(self.batch * self.N * 4),
                "matches_device_path": ok,
                "path": f"fft_stft_forward(host pinned signal / spectra): measured on {ch} of this rank's {self.channels} channels and scaled; unique samples uploaded once, 32 MiB chunks, H2D/kernel/D2H overlapped"}

    def cpu(self, seconds_target, steps=1, warmup=0):
        from oracle import oracle as o

        ref = o.load_ref()
        cores = min(ref.hardware_threads(), host_cores())
        rng = np.random.default_rng(42)
        # one channel per call: 934 overlapping frames split across the cores (out of place, frames overlap)
        xin = o.aligned_copy(rng.uniform(-1, 1, self.samples).astype(np.float32))
        out = o.aligned_empty(self.frames * self.N)
        run = lambda reps=1: ref.transform_timed(xin, out, self.N, False, False, True, self.frames, self.hop, self.N, cores, reps=reps)
        t1 = run()
        reps = max(1, int(seconds_target / max(t1, 1e-6) / max(1, steps + warmup)))
        times = [run(reps) for _ in range(warmup + steps)][warmup:]
        per_step = float(np.mean(times))
        bytes_ch = self.samples * 4 + self.frames * self.N * 4
        gbs = reps * bytes_ch / per_step / 1e9
        return gbs, cores, f"{reps} channels x 934 frames per step, {cores} threads, reference AVX build", per_step * 1e3


class ISTFT(STFT):
    """Inverse of BASELINE configs[2] (SURVEY.md §8f rank 1): overlap-add synthesis of 1024 channels x 934 frames of
    N=2048 at hop 512, Hann synthesis window, one fused kernel (C2R + window + overlap-add)."""

    def __init__(self):
        super().__init__()
        self.name = "istft"
        self.desc = "overlap-add synthesis (ISTFT): C2R N=2048 hop 512, 1024 channels x 934 frames, Hann window (inverse of BASELINE configs[2])"
        self.kernel = "cfb::istft_kernel<10,32,0>"

    def config(self):
        c = super().config()
        c.update({"transform": "C2R + overlap-add", "window": "Hann (synthesis)", "bytes": "packed spectra in + unique signal out"})
        return c

    def setup(self, cf, torch, rank, world):
        super().setup(cf, torch, rank, world)
        self.spec = torch.empty(self.channels, self.frames, self.N, device="cuda")
        cf.fft_transform_strided(self.plan, self.x, self.spec, self.channels, self.frames, self.samples, self.hop, self.frames * self.N, self.N, cf.FFT_FORWARD, True)
        n = torch.arange(self.N, device="cuda", dtype=torch.float64)
        self.win = (0.5 - 0.5 * torch.cos(2 * math.pi * (n + 0.5) / self.N)).float()
        self.out = torch.empty(self.channels, self.samples, device="cuda")
        del self.y

    def step(self, stream):
        self.cf.fft_istft_overlap_add(self.plan, self.spec, self.out, self.channels, self.frames, self.frames * self.N, self.N,
                                      self.samples, self.hop, self.win, 1.0 / self.N, True, stream)

    def outputs(self):
        return {"out": self.out}

    def parity(self):
        from oracle import oracle as o

        c = self.channels - 1
        want = o.np_istft_overlap_add(self.spec[c:c + 1].cpu().numpy(), self.N, self.hop, 8, True, self.win.cpu().numpy(), 1.0 / self.N)
        got = self.out[c:c + 1, :want.shape[1]].cpu().numpy()
        return {"rel_l2_vs_oracle": o.rel_l2(got, want), "tolerance": o.parity_tol(self.N), "transforms": self.frames}

    def cpu(self, seconds_target, steps=1, warmup=0):
        raise RuntimeError("no CPU leg for the synthesis workload (the reference has no overlap-add entry point)")


class Reverb(BatchedFFT):
    """BASELINE configs[3]: partitioned convolution, 2^16-tap IR, N=8192 blocks, 4096 channels; one step =
    one block (4096 new samples) for every channel through the fused kernel."""

    scaling = "strong"

    def __init__(self):
        self.name, self.N, self.P, self.channels_total = "reverb", 8192, 16, 4096
        self.B = self.N // 2
        self.is_complex, self.ordered = False, False
        self.desc = "partitioned convolution reverb: 2^16-tap per-channel IR, N=8192, 16 partitions, 4096 channels (BASELINE configs[3])"
        self.kernel = "cfb::pconv_kernel<12,3>"
        # SURVEY.md §8(d): window in 16384 (new samples only) + FDL write 32768 + 16 x (FDL + H read) + out 16384
        self.bytes_per_channel_block = 16384 + 32768 + 16 * 32768 + 16 * 32768 + 16384
        self.flops_per_channel_block = 2 * 2.5 * 8192 * 13 + 16 * 4096 * 8

    def config(self):
        return {"workload": self.desc, "N": self.N, "partitions": self.P, "channels": self.channels_total, "block": self.B,
                "ir": "per-channel, pre-transformed, unordered layout (2 GiB)", "fused": "R2C -> 16 x MAC -> C2R -> overlap-save discard in one kernel",
                "bytes": "1 114 112 B per channel-block (SURVEY.md §8d); the X_t spectrum is reused from registers, so actual traffic is 32 KiB lower",
                "l2_policy": "4.6 GB per step, far larger than L2", "sharding": "channels split contiguously across GPUs, no collectives"}

    def setup(self, cf, torch, rank, world):
        from chowdsp_fft_b200.sharding import shard_range

        self.cf, self.torch = cf, torch
        _, self.channels = shard_range(self.channels_total, rank, world)
        self.batch = self.channels
        self.bytes_step = self.channels * self.bytes_per_channel_block
        self.flops_step = self.channels * self.flops_per_channel_block
        self.plan = cf.fft_new_setup(self.N, cf.FFT_REAL, True)
        gen = torch.Generator(device="cuda").manual_seed(42 + rank)
        self.blocks = 64
        self.sig = torch.rand(self.channels, (self.blocks + 1) * self.B, device="cuda", generator=gen) * 2 - 1
        self.sig[:, :self.B] = 0  # the block before the first one
        ir_t = (torch.rand(self.channels * self.P, self.N, device="cuda", generator=gen) * 2 - 1) * 1e-3
        ir_t[:, self.B:] = 0
        self.h = torch.empty_like(ir_t)
        cf.fft_transform_batched(self.plan, ir_t, self.h, self.channels * self.P, self.N, self.N, cf.FFT_FORWARD, False)
        del ir_t
        self.fdl = torch.zeros(self.channels, self.P, self.N, device="cuda")
        self.out = torch.empty(self.channels, self.blocks * self.B, device="cuda")
        self.t = 0
        for _ in range(self.P):  # fill the delay line so that every timed step sums all 16 partitions
            self.step(None)

    def step(self, stream):
        t = self.t
        tb = t % self.blocks
        win = self.sig[:, tb * self.B:]
        out = self.out[:, tb * self.B:]
        self.cf.fft_partitioned_convolve_step(self.plan, win.data_ptr(), self.sig.shape[1], self.h, self.P * self.N, self.fdl, self.P * self.N,
                                              out.data_ptr(), self.out.shape[1], self.channels, self.P, t, 1.0 / self.N, stream)
        self.t += 1

    def outputs(self):
        """the block the last step produced for every channel"""
        tb = (self.t - 1) % self.blocks
        return {"out": self.out[:, tb * self.B:(tb + 1) * self.B]}

    def parity(self):
        """Last timed block of two channels against the oracle's composition of the same reference calls."""
        from oracle import oracle as o

        t = self.t - 1
        tb = t % self.blocks
        got, want = [], []
        for c in (0, self.channels - 1):
            fdl = self.fdl[c].cpu().numpy()
            h = self.h[c * self.P:(c + 1) * self.P].cpu().numpy()
            acc = np.zeros(self.N, np.float32)
            for p in range(self.P):
                acc = o.np_convolve(fdl[(t - p) % self.P], h[p], acc, self.N, False, 8, 1.0 / self.N)
            want.append(o.np_transform(acc, self.N, False, 8, True, False)[self.B:])
            got.append(self.out[c, tb * self.B:(tb + 1) * self.B].cpu().numpy())
        return {"rel_l2_vs_oracle": o.rel_l2(np.stack(got), np.stack(want)), "tolerance": 1e-5, "transforms": 2}

    def e2e(self, steps, barrier, reduce_max):
        """One block step with HOST audio: the new 4096 samples of every channel come from pinned host memory and the 4096
        output samples go back to it; the delay line and the IR spectra are the convolver's state and stay on the device
        (as they stay in RAM across calls in the reference's usage)."""
        cf, torch = self.cf, self.torch
        hin = torch.empty(self.channels, self.B, pin_memory=True)
        hout = torch.empty(self.channels, self.B, pin_memory=True)
        hin.copy_(self.sig[:, self.B:2 * self.B].cpu())
        win = torch.zeros(self.channels, self.N, device="cuda")
        dout = torch.empty(self.channels, self.B, device="cuda")
        st = torch.cuda.current_stream()

        def call():
            win[:, :self.B].copy_(win[:, self.B:], non_blocking=True)     # previous block slides down (device-local)
            win[:, self.B:].copy_(hin, non_blocking=True)                 # H2D: the new samples
            cf.fft_partitioned_convolve_step(self.plan, win, self.N, self.h, self.P * self.N, self.fdl, self.P * self.N, dout, self.B,
                                             self.channels, self.P, self.t, 1.0 / self.N, st)
            self.t += 1
            hout.copy_(dout, non_blocking=True)                           # D2H: the block's output
            torch.cuda.synchronize()
        call()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            call()
        dt = reduce_max((time.perf_counter() - t0) / steps)
        return {"seconds": dt, "h2d_bytes_per_step": int(self.channels * self.B * 4), "d2h_bytes_per_step": int(self.channels * self.B * 4),
                "matches_device_path": bool(torch.isfinite(hout).all()),
                "path": "pinned host block -> H2D -> fft_partitioned_convolve_step -> D2H, per block step; delay line + IR spectra resident on the device"}

    def cpu(self, seconds_target, steps=1, warmup=0):
        from oracle import oracle as o

        ref = o.load_ref()
        cores = min(ref.hardware_threads(), host_cores())
        channels, blocks = cores * 2, 48
        rng = np.random.default_rng(42)
        x = rng.uniform(-1, 1, (channels, blocks * self.B)).astype(np.float32)
        h = (rng.uniform(-1, 1, (channels, self.P, self.N)) * 1e-3).astype(np.float32)
        _, _, t1 = ref.partitioned_convolve(x, h, self.N, self.P, nthreads=cores)
        reps = max(1, int(seconds_target / max(t1, 1e-6) / max(1, steps + warmup)))
        times = []
        for it in range(warmup + steps):
            secs = 0.0
            for _ in range(reps):
                secs += ref.partitioned_convolve(x, h, self.N, self.P, nthreads=cores)[2]
            if it >= warmup:
                times.append(secs)
        per_step = float(np.mean(times))
        parts = sum(min(t + 1, self.P) for t in range(blocks))
        bytes_total = reps * channels * (blocks * (16384 + 32768 + 16384) + parts * 65536)
        gbs = bytes_total / per_step / 1e9
        return gbs, cores, f"{reps} x ({channels} channels x {blocks} blocks, {parts / blocks:.1f} partitions summed per block on average), {cores} threads, reference AVX build", per_step * 1e3


def hash_signal(torch, idx):
    """Counter-based synthetic signal keyed by the global FLOAT index (SURVEY.md §8d cfg 5: every GPU layout regenerates
    the same values): 64-bit LCG mix, top bits -> U(-1, 1).  idx: int64 tensor."""
    h = idx * 6364136223846793005 + 1442695040888963407
    h = (h ^ (h >> 29)) * 2862933555777941757 + 3037000493
    return ((h >> 40) & 0xFFFFFF).double() / float(1 << 23) - 1.0


def sampled_dft_of_hash_signal(torch, N, ks):
    """float64 DFT bins X[k] of the hash signal, phases from exact int64 arithmetic, chunked"""
    out = []
    step = 1 << 24
    for k in ks:
        re = im = 0.0
        for n0 in range(0, N, step):
            n = torch.arange(n0, min(N, n0 + step), device="cuda", dtype=torch.int64)
            ang = ((n * int(k)) % N).double() * (-2.0 * math.pi / N)
            c, sn = torch.cos(ang), torch.sin(ang)
            xr, xi = hash_signal(torch, 2 * n), hash_signal(torch, 2 * n + 1)
            re += float((xr * c - xi * sn).sum())
            im += float((xr * sn + xi * c).sum())
        out.append(complex(re, im))
    return np.array(out)


class Huge(BatchedFFT):
    """BASELINE configs[4]: ONE complex FFT of N = 2^28 points.  1 GPU: three-pass four-step on the device.
    G > 1 GPUs: distributed four-step through ONE C-ABI call per rank (fft_dist_transform): local tile passes, the
    all-to-all fused into phase 0's peer stores over NVLink, in-stream flag barrier; `natural` adds the second all-to-all
    (fused into the last pass's peer stores).  CFB_DIST_EXCHANGE=nccl times the NCCL all_to_all_single baseline instead."""

    scaling = "strong"

    def __init__(self, n=28, natural=False, exchange=None):
        self.name, self.n, self.N = "huge", n, 1 << n
        self.natural = natural
        self.exchange = exchange or os.environ.get("CFB_DIST_EXCHANGE", "peer")
        self.is_complex, self.ordered, self.nfl = True, True, 2 << n
        self.desc = f"single complex FFT N=2^{n} fp32 (BASELINE configs[4]): 3-pass four-step; distributed over G GPUs with the all-to-all over NVLink"
        self.kernel = "cfb::tile_fft_kernel<9|9|10> x3"
        self.phase_ms = None

    def config(self):
        c = {"workload": self.desc, "N": self.N, "transform": "C2C",
             "output": "natural order" if (self.world == 1 or self.natural) else "transposed-out per rank (one all-to-all)",
             "passes": 3, "bytes": "algorithmic 16 N = 4 GiB per transform; each of the 3 passes re-reads and re-writes the array",
             "l2_policy": "2 GiB arrays, far larger than L2", "sharding": "column blocks -> all-to-all -> row blocks"}
        if self.world > 1:
            c["exchange"] = self.exchange
            c["exchange_bytes_per_rank"] = self.d.exchange_bytes() * (2 if self.natural else 1)
        return c

    def setup(self, cf, torch, rank, world):
        self.cf, self.torch, self.rank, self.world = cf, torch, rank, world
        self.batch = 1
        self.bytes_step = 16 * self.N // world
        self.flops_step = 5.0 * self.N * math.log2(self.N) / world
        if world == 1:
            self.plan = cf.fft_new_setup(self.N, cf.FFT_COMPLEX, True)
            self.x = torch.empty(2 * self.N, device="cuda")
            step = 1 << 26
            for f0 in range(0, 2 * self.N, step):
                self.x[f0:f0 + step] = hash_signal(torch, torch.arange(f0, f0 + step, device="cuda", dtype=torch.int64)).float()
            self.y = torch.empty_like(self.x)
        else:
            from chowdsp_fft_b200.distributed import DistributedFFT

            self.d = d = DistributedFFT(self.n, rank, world, exchange=self.exchange)
            self.x = torch.empty(d.L1, d.cols, 2, device="cuda")
            rows = max(1, (1 << 24) // d.cols)
            c = torch.arange(d.cols, device="cuda", dtype=torch.int64)[None, :]
            for r0 in range(0, d.L1, rows):  # global complex index of every element of this rank's column block
                n1 = torch.arange(r0, min(d.L1, r0 + rows), device="cuda", dtype=torch.int64)[:, None]
                g = n1 * d.S1 + rank * d.cols + c
                self.x[r0:r0 + rows, :, 0] = hash_signal(torch, 2 * g).float()
                self.x[r0:r0 + rows, :, 1] = hash_signal(torch, 2 * g + 1).float()
            self.y = torch.empty(2 * (self.N // world), device="cuda")

    def step(self, stream):
        if self.world == 1:
            self.cf.fft_transform_batched(self.plan, self.x, self.y, 1, 2 * self.N, 2 * self.N, self.cf.FFT_FORWARD, True, stream)
        else:
            # natural order with the peer exchange: the result stays in the context's natural-order block (the one the
            # peers store into); no copy into a caller buffer inside the timed region
            out = None if (self.natural and self.exchange == "peer") else self.y
            self.d.forward(self.x, out, stream=stream, natural=self.natural)

    def outputs(self):
        """complex bins as rows of (re, im)"""
        # the natural-order peer exchange leaves its result in the distributed context, not in self.y
        assert not (self.natural and self.exchange == "peer"), "no caller-visible output to dump for this variant"
        return {"y": self.y.view(-1, 2)}

    def after_timing(self):
        """one extra, event-timed transform for the per-phase split (peer exchange only); it also fills self.y for the parity gate"""
        if self.world > 1 and self.exchange == "peer":
            import torch.distributed as dist

            torch = self.torch
            torch.cuda.synchronize()
            dist.barrier()  # every rank starts its phase 0 together: the exchange is timed under the full all-to-all load
            self.d.forward(self.x, self.y, natural=self.natural, timed=True)
            t = torch.tensor(self.d.phase_ms(), device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)  # slowest rank per phase
            self.phase_ms = [float(v) for v in t.tolist()]

    def nvlink(self):
        """G > 1: the exchange is the bound (SURVEY.md §8d cfg 5): bytes this rank sends in the fused phase 0 / its duration"""
        if self.world == 1 or not self.phase_ms:
            return None
        sent = self.d.exchange_bytes()
        window_ms = self.phase_ms[0] + self.phase_ms[1]
        gbs = sent / (window_ms * 1e-3) / 1e9
        return {"bound": "nvlink", "achieved": gbs, "peak": 900.0, "unit": "GB/s", "frac": gbs / 900.0, "frac_of_measured_peer_copy_770": gbs / 770.0,
                "traffic": None, "exchange_bytes_per_rank": sent, "exchange_window_ms": window_ms,
                "phase_ms": {"phase0_fft_plus_peer_stores": self.phase_ms[0], "flag_barrier_wait": self.phase_ms[1], "phases_1_2_local": self.phase_ms[2],
                             "natural_order_barrier_and_copy": self.phase_ms[3]},
                "kernel": "cfb::tile_fft_kernel (phase 0, peer-store epilogue) + cfb::dist_barrier_kernel",
                "peak_source": "nominal NVLink 5 per direction per GPU (B200_PROFILING.md; measured peer copy 770 GB/s)"}

    def parity(self):
        torch = self.torch
        rng = np.random.default_rng(7 + self.rank)
        if self.world == 1:
            ks = sorted(set([0, 1, self.N - 1, self.N // 2] + [int(k) for k in rng.integers(0, self.N, 12)]))
            got = self.y.view(-1, 2)[torch.tensor(ks, device="cuda")].cpu().numpy()
        elif self.natural or self.exchange == "nccl" and False:
            blk = self.N // self.world
            idx = [int(i) for i in rng.integers(0, blk, 8)]
            ks = [self.rank * blk + i for i in idx]
            got = self.y.view(-1, 2)[torch.tensor(idx, device="cuda")].cpu().numpy()
        else:
            d = self.d
            qs, kk = rng.integers(0, d.S1, 8), rng.integers(0, d.rows, 8)
            ks = [int(self.rank * d.rows + k + d.L1 * q) for q, k in zip(qs, kk)]
            got = self.y.view(d.S1, d.rows, 2)[torch.tensor(qs, device="cuda"), torch.tensor(kk, device="cuda")].cpu().numpy()
        want = sampled_dft_of_hash_signal(torch, self.N, ks)
        got = got[:, 0].astype(np.float64) + 1j * got[:, 1]
        return {"rel_l2_vs_float64_dft": float(np.linalg.norm(got - want) / np.linalg.norm(want)), "tolerance": 1e-6 * self.n, "bins": len(ks),
                "note": "rank 0's share of the spectrum, sampled bins against a float64 DFT with exact integer phases"}

    def e2e(self, steps, barrier, reduce_max):
        if self.world != 1:
            return None
        return BatchedFFT.e2e(self, steps, barrier, reduce_max)

    def cpu(self, seconds_target, steps=1, warmup=0):
        """The reference cannot thread one transform: 1 core by construction (SURVEY.md §8d); bounded to 2^24."""
        from oracle import oracle as o

        ref = o.load_ref()
        n = 24
        N = 1 << n
        rng = np.random.default_rng(42)
        xin = o.aligned_copy(rng.uniform(-1, 1, 2 * N).astype(np.float32))
        out = o.aligned_empty(2 * N)
        times = []
        for it in range(warmup + steps):
            times.append(ref.transform_timed(xin, out, N, True, False, True, 1, 2 * N, 2 * N, 1))
        per = float(np.mean(times[warmup:] or times))
        return 16 * N / per / 1e9, 1, f"one C2C N=2^{n} transform (plan setup excluded), 1 thread: the reference is single-threaded per transform", per * 1e3


class Single1024(BatchedFFT):
    """BASELINE configs[0]: ONE real FFT N=1024, forward + inverse round trip through the drop-in calls (the
    reference's own bench loop, bench/bench.cpp:82-110).  A latency case: the line's value is still GB/s, the
    numbers that matter are in config.latency_us (sync call, stream-ordered, CUDA-graph replay)."""

    scaling = "weak"

    def __init__(self):
        BatchedFFT.__init__(self, "single1024", 1024, False, 1, True, "single real FFT N=1024 forward+inverse round trip fp32 (BASELINE configs[0])")
        self.bytes_step = 2 * 8 * self.N
        self.flops_step = 2 * 2.5 * self.N * math.log2(self.N)
        self.kernel = "cfb::fft_kernel<9,16,R2C,0> + cfb::fft_kernel<9,16,C2R,0>"
        self.latency = {}

    def config(self):
        c = BatchedFFT.config(self)
        c["l2_policy"] = "latency case: 4 KiB buffers, cache-resident by construction (as in the reference's bench loop)"
        c["latency_us"] = self.latency
        return c

    def setup(self, cf, torch, rank, world):
        self.cf, self.torch = cf, torch
        self.plan = cf.fft_new_setup(self.N, cf.FFT_REAL, True)
        i = torch.arange(self.N, device="cuda", dtype=torch.float32)
        self.x = torch.sin(3.14 * (100.0 / 48000.0) * i).reshape(1, self.N)  # bench/bench.cpp:82-85
        self.y = torch.empty_like(self.x)
        self.z = torch.empty_like(self.x)
        self.step(None)
        torch.cuda.synchronize()
        # (1) the drop-in calls: synchronous on return, like the reference's
        t0 = time.perf_counter()
        for _ in range(200):
            cf.fft_transform(self.plan, self.x, self.y, None, cf.FFT_FORWARD)
            cf.fft_transform(self.plan, self.y, self.z, None, cf.FFT_BACKWARD)
        self.latency["drop_in_sync_calls"] = (time.perf_counter() - t0) / 200 * 1e6
        # (1b) the same loop as a COMPILED C caller (tests/c_caller/latency_bench.c = the reference's bench/bench.cpp loop on
        # aligned_malloc buffers): the latency of the drop-in calls without the ctypes binding around them
        self.latency["drop_in_sync_calls_compiled_c_caller"] = self.c_caller_latency("1")
        self.latency["drop_in_sync_calls_compiled_c_caller_blocking_sync"] = self.c_caller_latency("0")
        # (2) CUDA-graph replay of 100 round trips
        side = torch.cuda.Stream()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.stream(side):
            with torch.cuda.graph(g, stream=side):
                for _ in range(100):
                    self.step(side)
            g.replay()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(side)
            for _ in range(10):
                g.replay()
            e1.record(side)
            torch.cuda.synchronize()
        self.latency["cuda_graph_replay"] = e0.elapsed_time(e1) / 1000 * 1e3
        self.graph = g

    def c_caller_latency(self, spin):
        import subprocess
        import tempfile

        from chowdsp_fft_b200 import _lib

        try:
            exe = os.path.join(tempfile.gettempdir(), "cfb_latency_bench")
            src = os.path.join(ROOT, "tests", "c_caller", "latency_bench.c")
            r = subprocess.run(["gcc", "-std=c11", "-O2", f"-I{os.path.join(ROOT, 'include')}", src, _lib.LIB_PATH, f"-Wl,-rpath,{os.path.dirname(_lib.LIB_PATH)}", "-lm", "-o", exe],
                               capture_output=True, text=True, timeout=120)
            if r.returncode != 0:
                return None
            r = subprocess.run([exe, str(self.N), "2000"], capture_output=True, text=True, timeout=120, env=dict(os.environ, CHOWDSP_FFT_B200_SPIN_SYNC=spin))
            tok = r.stdout.split()
            return float(tok[tok.index("us_per_round_trip") + 1]) if r.returncode == 0 else None
        except Exception:
            return None

    def step(self, stream):
        cf = self.cf
        cf.fft_transform_batched(self.plan, self.x, self.y, 1, self.N, self.N, cf.FFT_FORWARD, True, stream)
        cf.fft_transform_batched(self.plan, self.y, self.z, 1, self.N, self.N, cf.FFT_BACKWARD, True, stream)

    def outputs(self):
        return {"y": self.y, "z": self.z}

    def parity(self):
        from oracle import oracle as o

        x = self.x.cpu().numpy()
        f = o.np_transform(x, self.N, False, 8, False, True)
        return {"rel_l2_vs_oracle": max(o.rel_l2(self.y.cpu().numpy(), f), o.rel_l2(self.z.cpu().numpy() / self.N, x)),
                "tolerance": o.parity_tol(self.N), "transforms": 2}

    def e2e(self, steps, barrier, reduce_max):
        cf = self.cf
        hin, hmid, hout = cf.aligned_array(self.N), cf.aligned_array(self.N), cf.aligned_array(self.N)
        hin[:] = self.x.cpu().numpy()[0]
        n = 200
        def call():
            cf.fft_transform(self.plan, hin, hmid, None, cf.FFT_FORWARD)
            cf.fft_transform(self.plan, hmid, hout, None, cf.FFT_BACKWARD)
        call()
        t0 = time.perf_counter()
        for _ in range(n):
            call()
        dt = (time.perf_counter() - t0) / n
        self.latency["drop_in_host_buffers"] = dt * 1e6
        ok = bool(np.allclose(hout / self.N, hin, atol=1e-5))
        for h in (hin, hmid, hout):
            cf.aligned_free(h.ctypes.data)
        return {"seconds": dt, "h2d_bytes_per_step": 2 * 4 * self.N, "d2h_bytes_per_step": 2 * 4 * self.N, "matches_device_path": ok,
                "path": "fft_transform x2 on aligned_malloc (pinned, device-mapped) host buffers: zero-copy kernel, one sync per call"}

    def cpu(self, seconds_target, steps=1, warmup=0):
        from oracle import oracle as o

        ref = o.load_ref()
        xin = o.aligned_copy(np.sin(3.14 * (100.0 / 48000.0) * np.arange(self.N)).astype(np.float32))
        out, back = o.aligned_empty(self.N), o.aligned_empty(self.N)
        reps = 20000
        times = []
        for it in range(warmup + max(1, steps)):
            t = 0.0
            for _ in range(4):
                t += ref.transform_timed(xin, out, self.N, False, False, True, reps, 0, 0, 1)
                t += ref.transform_timed(out, back, self.N, False, True, True, reps, 0, 0, 1)
            times.append(t / 4)
        per = float(np.mean(times[warmup:] or times)) / reps  # one forward + one backward
        self.latency["reference_cpu_1_thread"] = per * 1e6
        return self.bytes_step / per / 1e9, 1, f"{reps} forward + {reps} backward transforms of the same 4 KiB buffer per step, 1 thread (reference bench loop)", per * reps * 1e3


WORKLOADS = {
    "istft": ISTFT,
    "c2c4096": lambda: BatchedFFT("c2c4096", 4096, True, 65536, True, "batched C2C N=4096 x 65536 fp32, ordered, forward (BASELINE configs[1])"),
    "c2c4096_unordered": lambda: BatchedFFT("c2c4096_unordered", 4096, True, 65536, False, "batched C2C N=4096 x 65536 fp32, unordered (reference W=8 layout), forward (BASELINE configs[1])"),
    "c2c1024": lambda: BatchedFFT("c2c1024", 1024, True, 262144, True, "batched C2C N=1024 x 262144 fp32, ordered, forward"),
    "c2c8192": lambda: BatchedFFT("c2c8192", 8192, True, 32768, True, "batched C2C N=8192 x 32768 fp32, ordered, forward"),
    "c2c16384": lambda: BatchedFFT("c2c16384", 16384, True, 16384, True, "batched C2C N=16384 x 16384 fp32, ordered, forward"),
    "c2c16384_unordered": lambda: BatchedFFT("c2c16384_unordered", 16384, True, 16384, False, "batched C2C N=16384 x 16384 fp32, unordered, forward"),
    "r2c2048": lambda: BatchedFFT("r2c2048", 2048, False, 524288, True, "batched R2C N=2048 x 524288 fp32, ordered, forward"),
    "r2c8192": lambda: BatchedFFT("r2c8192", 8192, False, 131072, False, "batched R2C N=8192 x 131072 fp32, unordered, forward"),
    "single1024": Single1024,
    "stft": STFT,
    "reverb": Reverb,
    "huge": Huge,
}


def load_traffic(name, kernel_name):
    """ncu dram bytes per launch of the dominant kernel, from the committed capture summary -- only if that capture was of
    the kernel this run was actually routed to (otherwise null: a stale figure must not ride along silently)"""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            ent = json.load(f).get(name)
    except Exception:
        return None, None
    if not isinstance(ent, dict):
        return None, None
    if ent.get("kernel") and ent["kernel"] not in kernel_name:
        return None, f"capture was of {ent['kernel']}, this run used {kernel_name}"
    return ent.get("bytes"), ent.get("source")


DUMP_BYTES = 64_000_000  # --dump-outputs writes at most this much in all


def dump_outputs(torch, outputs, out_dir):
    """Writes every output as out_dir/<name>.npy (float32).  An output larger than its share of DUMP_BYTES is cut down to
    a sample of its rows that depends only on its shape (the same rows on every run, in row order), so that two builds
    run with the same arguments can be compared array for array."""
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // len(outputs)
    for name, t in outputs.items():
        if t.numel() * 4 > share:
            rows = t.reshape(-1, t.shape[-1])
            keep = share // (rows.shape[1] * 4)
            idx = np.unique(np.random.default_rng(0).integers(0, rows.shape[0], keep))
            t = rows[torch.from_numpy(idx).to(rows.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def measure(wl, name, ctx, steps, warmup, do_e2e, do_cpu, cpu_seconds, tune=None, dump_dir=None):
    """warm-up, `steps` timed steps (CUDA events on the launch stream, barrier + synchronize on both sides, max over
    ranks), outputs of the last step to `dump_dir` (rank 0), parity check, e2e with host buffers, CPU baseline -> one
    record"""
    cf, torch, dist = ctx["cf"], ctx["torch"], ctx["dist"]
    rank, world, local_rank = ctx["rank"], ctx["world"], ctx["local_rank"]
    barrier, reduce_max, reduce_sum = ctx["barrier"], ctx["reduce_max"], ctx["reduce_sum"]
    wl.setup(cf, torch, rank, world)
    stream = torch.cuda.current_stream()
    for _ in range(max(3, warmup)):
        wl.step(stream)
    barrier()
    launches0 = cf.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:
        ev0.record(stream)
        for _ in range(steps):
            wl.step(stream)
        ev1.record(stream)
        barrier()
    launches = cf.launch_count() - launches0
    kernel_name = cf.last_kernel() or wl.kernel  # what the library actually routed this workload to
    ms_local = ev0.elapsed_time(ev1) / steps
    ms_step = reduce_max(ms_local)
    bytes_job = reduce_sum(float(wl.bytes_step))
    flops_job = reduce_sum(float(wl.flops_step))
    value = bytes_job / (ms_step * 1e-3) / 1e9
    per_gpu = wl.bytes_step / (ms_local * 1e-3) / 1e9
    peak, peak_src = hbm_peak()
    if dump_dir is not None and rank == 0:
        dump_outputs(torch, wl.outputs(), dump_dir)
    if hasattr(wl, "after_timing"):
        wl.after_timing()

    parity = None
    if rank == 0:
        try:
            parity = wl.parity()  # quick gate beside the timing; tests/ hold the real parity suite
        except Exception as e:
            parity = {"error": repr(e)}
    e2e = None
    if do_e2e:
        r = wl.e2e(max(2, min(5, steps)), barrier, reduce_max)
        if r is not None:
            secs = r.pop("seconds")
            e2e = {"value": bytes_job / secs / 1e9, "unit": "GB/s", "ms_per_step": secs * 1e3, **r}
    cpu = None
    if rank == 0 and do_cpu:
        try:
            gbs, cores, desc, _ = wl.cpu(seconds_target=cpu_seconds)
            cpu = {"value": gbs, "unit": "GB/s", "cores": cores, "kind": "reference", "sample": desc}
        except Exception as e:
            cpu = {"value": None, "unit": "GB/s", "cores": 0, "kind": "reference", "sample": f"unavailable: {e!r}"}
    traffic, traffic_src = load_traffic(name, kernel_name)
    roofline = {"bound": "hbm", "achieved": per_gpu, "peak": peak, "unit": "GB/s", "frac": per_gpu / peak,
                "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "frac_of_nominal_8TBs": per_gpu / 8000.0,
                "kernel": kernel_name, "algorithmic_bytes_per_step": wl.bytes_step, "launches_per_step": launches / max(1, steps)}
    nv = wl.nvlink() if hasattr(wl, "nvlink") else None
    if nv is not None:
        nv["hbm_view"] = roofline
        roofline = nv
    rec = {"metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": world, "steps": steps, "warmup": max(3, warmup),
           "ms_per_step": ms_step, "higher_is_better": True, "scaling": wl.scaling, "vs_baseline": None, "dtype": "f32",
           "data": "synthetic", "config": wl.config(), "gflops": flops_job / (ms_step * 1e-3) / 1e9, "roofline": roofline,
           "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks.summary(), "parity": parity}
    if tune:
        rec["config"]["tuning"] = tune
    return rec


def release(wl, torch):
    for k in list(vars(wl)):
        v = getattr(wl, k)
        if hasattr(v, "close") and k == "d":
            v.close()
        if torch.is_tensor(v):
            delattr(wl, k)
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps of the headline and of every sub-record (the e2e leg with host buffers times max(2, min(5, K)) calls)")
    ap.add_argument("--warmup", type=int, default=3, help="warm-up steps before the timed ones, at least 3 whatever the value")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS), help="one workload only (default: the headline c2c4096 plus sub-records of every BASELINE config)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="headline workload only, no per-config sub-records")
    ap.add_argument("--tune", action="append", default=[], metavar="KEY=VALUE", help="fft_b200_set_tuning hook (sweeps only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the headline workload's outputs of its last timed step as DIR/<name>.npy (float32, at most 64 MB "
                         "in all: a fixed sample of rows of larger outputs); inputs are seeded, so runs with the same arguments compare. "
                         "With --gpus > 1, rank 0's share only, in the layout its step leaves it")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path computed; the reference arm has no such outputs")
    headline = args.workload or "c2c4096"
    wl = WORKLOADS[headline]()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    # ---------------------------------------------------------------- reference arm (CPU, rank 0 only)
    if args.impl == "reference":
        if rank != 0:
            return
        wl.world = 1
        gbs, cores, desc, ms = wl.cpu(seconds_target=20.0, steps=max(1, args.steps), warmup=args.warmup)
        flops_per_byte = (5.0 * wl.N * math.log2(wl.N)) / (16 * wl.N) if wl.is_complex else None
        line = {"impl": "reference", "metric": METRIC, "value": gbs, "unit": "GB/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
                "scaling": wl.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": wl.config(),
                "gflops": gbs * flops_per_byte if flops_per_byte else None,
                "cpu_baseline": {"value": gbs, "unit": "GB/s", "cores": cores, "kind": "reference", "sample": desc},
                "e2e": {"value": gbs, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    # ---------------------------------------------------------------- our arm
    import torch
    import torch.distributed as dist

    import chowdsp_fft_b200 as cf

    if not torch.cuda.is_available() or not cf.device_available():
        raise SystemExit("bench.py: no CUDA device; chowdsp_fft_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce(v, op):
        t = torch.tensor([v], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=op)
        return float(t.item())

    ctx = {"cf": cf, "torch": torch, "dist": dist, "rank": rank, "world": world, "local_rank": local_rank, "barrier": barrier,
           "reduce_max": lambda v: reduce(v, dist.ReduceOp.MAX), "reduce_sum": lambda v: reduce(v, dist.ReduceOp.SUM)}
    for kv in args.tune:
        k, v = kv.split("=")
        cf.set_tuning(k, int(v, 0))
    t_start = time.perf_counter()
    line = measure(wl, headline, ctx, args.steps, args.warmup, not args.no_e2e, world == 1 and not args.no_cpu, 12.0, args.tune,
                   args.dump_outputs)
    release(wl, torch)

    # ---------------------------------------------------------------- sub-records: every BASELINE config in the driver-run line
    if args.workload is None and not args.no_configs:
        subs = []
        if world == 1:
            plan = [("configs[0] single real N=1024 round trip (latency)", "single1024", Single1024),
                    ("configs[1] unordered half", "c2c4096_unordered", WORKLOADS["c2c4096_unordered"]),
                    ("configs[2] STFT", "stft", STFT),
                    ("configs[3] reverb", "reverb", Reverb),
                    ("configs[4] N=2^28 on one GPU", "huge", Huge)]
        else:
            plan = [("configs[2] STFT, channels sharded (strong scaling)", "stft", STFT),
                    ("configs[4] N=2^28 distributed, fused peer exchange, transposed-out", "huge", lambda: Huge(exchange="peer")),
                    ("configs[4] N=2^28 distributed, fused peer exchange, natural order (second all-to-all fused)", "huge", lambda: Huge(natural=True, exchange="peer")),
                    ("configs[4] N=2^28 distributed, NCCL all_to_all_single baseline, transposed-out", "huge", lambda: Huge(exchange="nccl"))]
        for label, name, make in plan:
            try:
                w = make()
                rec = measure(w, name, ctx, args.steps, args.warmup, not args.no_e2e, world == 1 and not args.no_cpu, 3.0)
                rec["baseline_config"] = label
                release(w, torch)
            except Exception as e:  # a sub-record must not take the headline down
                rec = {"baseline_config": label, "error": repr(e)}
            subs.append(rec)
        line["configs"] = subs
    line["bench_wall_seconds"] = time.perf_counter() - t_start
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
