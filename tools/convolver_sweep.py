#!/usr/bin/env python
"""Streaming convolver (fft_convolver_process, non-uniform partitions) against the uniform fused step
(fft_partitioned_convolve_step with P = L / B partitions of block B) at the same (B, L, channels), per-channel and shared IR.

For each configuration, after one warm-up period, it alternates REPS times: one full period of the convolver (Bmax / B calls,
so every segment fires at its average rate) and the same number of uniform steps.  Every call is timed alone with CUDA events
on the stream; the table gives mean and max per-call times.  A call's time includes any gap the host leaves between its launches
(the convolver makes 3-5 launches per call), so small channel counts measure launch overhead, not bandwidth.

Algorithmic bytes per input sample and channel, HBM traffic as the kernels are written (delay-line and IR reads 16 P_k per segment,
window 8, delay-line write 8, output / accumulator 8-12, input history 12, tail partial spectrum 16; a shared IR counted once per
step across channels).  Working sets are 0.3-4 GiB, larger than L2 except for the shared-IR cases at 256 channels.
GPU only: prints the card name and power limit next to the numbers."""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
import torch

import chowdsp_fft_b200 as cf

BMAX = 16384


def uniform_bytes(B, L, channels, shared):
    P = -(-L // B)
    ir = 8 * P / channels if shared else 8 * P
    return 8 * P + ir + 20


def convolver_bytes(segs, B, channels, shared):
    total = 12.0  # input history: read 4, two writes
    for k, (bk, p) in enumerate(segs):
        ir = 8 * p / channels if shared else 8 * p
        total += 8 * p + ir + 8 + 8 + (12 if k == 0 else 8)
    if len(segs) > 1 and segs[-1][1] > 1:
        total += 16
    return total


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        q = "power limit not available"
    return f"{name}, {q}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--blocks", type=int, nargs="*", default=[128, 512])
    ap.add_argument("--lengths", type=int, nargs="*", default=[1 << 16, 1 << 18])
    ap.add_argument("--channels", type=int, nargs="*", default=[256, 1024])
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    st = torch.cuda.current_stream()
    print(f"# {card()}", flush=True)
    print(f"# {'B':>5} {'L':>7} {'ch':>5} {'ir':>7} | {'conv B/smp':>10} {'mean ms':>8} {'max ms':>8} | {'unif B/smp':>10} {'mean ms':>8} "
          f"{'max ms':>8} | {'mean ratio':>10} {'max ratio':>9} | segments", flush=True)
    for B in args.blocks:
        for L in args.lengths:
            for channels in args.channels:
                for shared in (False, True):
                    g = torch.Generator(device="cuda").manual_seed(B + L + channels)
                    D = BMAX // B
                    nir = 1 if shared else channels
                    ir = torch.rand(nir, L, device="cuda", generator=g) / L
                    ctx = cf.fft_convolver_create(channels, B, ir, L, 0 if shared else L)
                    segs = cf.fft_convolver_segments(ctx)
                    del ir
                    x = torch.rand(channels, B, device="cuda", generator=g) * 2 - 1
                    y = torch.empty(channels, B, device="cuda")
                    # uniform step: random spectra stand in for the IR (timing only)
                    N, P = 2 * B, -(-L // B)
                    s = cf.fft_new_setup(N, cf.FFT_REAL)
                    hspec = torch.rand(nir, P, N, device="cuda", generator=g) * 1e-3
                    fdl = torch.zeros(channels, P, N, device="cuda")
                    win = torch.rand(channels, N, device="cuda", generator=g)
                    out = torch.empty(channels, B, device="cuda")
                    step = [P]  # steady state from the first call: every partition is summed

                    def conv_call():
                        cf.fft_convolver_process(ctx, x, B, y, B, st)

                    def unif_call():
                        cf.fft_partitioned_convolve_step(s, win, N, hspec, 0 if shared else P * N, fdl, P * N, out, B, channels, P, step[0], 1.0 / N, st)
                        step[0] += 1

                    def timed(fn, n):
                        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
                        for a, b in ev:
                            a.record(st)
                            fn()
                            b.record(st)
                        torch.cuda.synchronize()
                        return [a.elapsed_time(b) for a, b in ev]

                    timed(conv_call, D)
                    timed(unif_call, D)
                    tc, tu = [], []
                    for _ in range(args.reps):
                        tc += timed(conv_call, D)
                        tu += timed(unif_call, D)
                    mc, xc, mu, xu = sum(tc) / len(tc), max(tc), sum(tu) / len(tu), max(tu)
                    print(f"  {B:5d} {L:7d} {channels:5d} {'shared' if shared else 'per-ch':>7} | {convolver_bytes(segs, B, channels, shared):10.0f} "
                          f"{mc:8.4f} {xc:8.4f} | {uniform_bytes(B, L, channels, shared):10.0f} {mu:8.4f} {xu:8.4f} | {mc / mu:10.3f} {xc / mu:9.3f} | "
                          f"{' '.join(f'{b}x{p}' for b, p in segs)}", flush=True)
                    cf.fft_convolver_destroy(ctx)
                    cf.fft_destroy_setup(s)
                    del x, y, hspec, fdl, win, out
                    torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
