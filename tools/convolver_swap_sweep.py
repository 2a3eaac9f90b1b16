#!/usr/bin/env python
"""Cost of replacing the streaming convolver's IR on a live context (fft_convolver_set_ir), at the configurations of
tools/convolver_sweep.py (DESIGN.md §3.4b), per-channel and shared IR.

For each configuration, after one warm-up period and the first set_ir (which allocates the second IR bank, untimed), it
repeats REPS times: one period of plain calls (Bmax / B calls, every segment fires at its average rate), an instant set_ir,
a set_ir with a crossfade over one full period followed by that period of fading calls, and one period of plain calls after
the swap.  Device times come from CUDA events on the stream around each call; the set_ir host column is the time the call
takes to return (it queues work and does not synchronise).  set_ir runs after the largest segment's first firing, so its
re-prime re-runs one firing of every segment.  GPU only: prints the card name and power limit next to the numbers."""
import argparse
import os
import sys
import time

sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
import torch

import chowdsp_fft_b200 as cf
from convolver_sweep import BMAX, card


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--blocks", type=int, nargs="*", default=[128, 512])
    ap.add_argument("--lengths", type=int, nargs="*", default=[1 << 16, 1 << 18])
    ap.add_argument("--channels", type=int, nargs="*", default=[256, 1024])
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    st = torch.cuda.current_stream()
    print(f"# {card()}", flush=True)
    print(f"# {'B':>5} {'L':>7} {'ch':>5} {'ir':>7} | {'plain mean':>10} {'max ms':>8} | {'set_ir ms':>9} {'host ms':>8} | {'fade mean':>9} "
          f"{'max ms':>8} | {'after mean':>10} {'max ms':>8} | {'fade/plain':>10}", flush=True)
    for B in args.blocks:
        for L in args.lengths:
            for channels in args.channels:
                for shared in (False, True):
                    g = torch.Generator(device="cuda").manual_seed(B + L + channels)
                    D = BMAX // B
                    nir = 1 if shared else channels
                    stride = 0 if shared else L
                    irs = [torch.rand(nir, L, device="cuda", generator=g) / L for _ in range(2)]
                    ctx = cf.fft_convolver_create(channels, B, irs[0], L, stride)
                    x = torch.rand(channels, B, device="cuda", generator=g) * 2 - 1
                    y = torch.empty(channels, B, device="cuda")

                    def conv_call():
                        cf.fft_convolver_process(ctx, x, B, y, B, st)

                    def timed(fn, n):
                        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
                        for a, b in ev:
                            a.record(st)
                            fn()
                            b.record(st)
                        torch.cuda.synchronize()
                        return [a.elapsed_time(b) for a, b in ev]

                    timed(conv_call, D)
                    cf.fft_convolver_set_ir(ctx, irs[0], L, stride, 0, st)  # allocates the second bank
                    timed(conv_call, D // 2)  # swaps below land mid-period
                    plain, sets, host, fade, after = [], [], [], [], []
                    nxt = 1
                    for _ in range(args.reps):
                        plain += timed(conv_call, D)
                        for fade_blocks in (0, D):
                            def set_call():
                                h0 = time.perf_counter()
                                cf.fft_convolver_set_ir(ctx, irs[nxt], L, stride, fade_blocks, st)
                                host.append((time.perf_counter() - h0) * 1e3)

                            sets += timed(set_call, 1)
                            nxt ^= 1
                            if fade_blocks:
                                fade += timed(conv_call, D)
                        after += timed(conv_call, D)
                    mean = lambda v: sum(v) / len(v)
                    print(f"  {B:5d} {L:7d} {channels:5d} {'shared' if shared else 'per-ch':>7} | {mean(plain):10.4f} {max(plain):8.4f} | "
                          f"{mean(sets):9.3f} {mean(host):8.3f} | {mean(fade):9.4f} {max(fade):8.4f} | {mean(after):10.4f} {max(after):8.4f} | "
                          f"{mean(fade) / mean(plain):10.2f}", flush=True)
                    cf.fft_convolver_destroy(ctx)
                    del irs, x, y
                    torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
