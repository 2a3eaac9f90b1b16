#!/usr/bin/env python
"""Cost of the streaming STFT contexts (fft_stft_stream_analyze / fft_stft_stream_synthesize, DESIGN.md §3.5b) per call, against
the offline calls over the same total frames, and the headroom against real time.

For each N / hop, channel count and frames per call F: a context with Hann windows and ordered spectra; CALLS analyze calls and
CALLS synthesize calls after a warm-up, each timed alone by CUDA events on the stream (mean and max in ms).  The offline column
times fft_stft_forward / fft_istft_overlap_add (default routing) on TOTAL frames per channel, best of 3 calls; the ratio is
(per-call time x TOTAL / F) over that offline time.  Headroom = the duration of F hops at 48 kHz over the time of one analyze
plus one synthesize call.  GPU only: prints the card name and power limit next to the numbers."""
import argparse
import os
import sys

sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
import torch

import chowdsp_fft_b200 as cf
from convolver_sweep import card


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", nargs="*", default=["2048/512", "1024/256", "512/128"])
    ap.add_argument("--channels", type=int, nargs="*", default=[64, 1024, 4096])
    ap.add_argument("--frames", type=int, nargs="*", default=[1, 16])
    ap.add_argument("--calls", type=int, default=100)
    ap.add_argument("--total", type=int, default=128, help="frames per channel of the offline calls")
    args = ap.parse_args()
    st = torch.cuda.current_stream()

    def timed(fn, n):
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
        for a, b in ev:
            a.record(st)
            fn()
            b.record(st)
        torch.cuda.synchronize()
        return [a.elapsed_time(b) for a, b in ev]

    print(f"# {card()}", flush=True)
    print(f"# {'N/hop':>9} {'ch':>5} {'F':>3} | {'analyze ms':>10} {'max':>7} {'offline ms':>10} {'ratio':>6} | {'synth ms':>9} {'max':>7} "
          f"{'offline ms':>10} {'ratio':>6} | {'budget ms':>9} {'headroom':>8}", flush=True)
    for cfg in args.configs:
        N, hop = (int(v) for v in cfg.split("/"))
        s = cf.fft_new_setup(N, cf.FFT_REAL)
        win = 0.5 - 0.5 * torch.cos(2 * torch.pi * torch.arange(N, device="cuda") / N)
        for channels in args.channels:
            T = args.total
            g = torch.Generator(device="cuda").manual_seed(N + channels)
            sig = torch.rand(channels, (T - 1) * hop + N, device="cuda", generator=g) * 2 - 1
            spec_all = torch.empty(channels, T, N, device="cuda")
            cf.fft_stft_forward(s, sig, spec_all, channels, T, sig.shape[1], hop, T * N, N, win, True, st)
            off_a = min(timed(lambda: cf.fft_stft_forward(s, sig, spec_all, channels, T, sig.shape[1], hop, T * N, N, win, True, st), 3))
            out_all = torch.empty_like(sig)
            off_s = min(timed(lambda: cf.fft_istft_overlap_add(s, spec_all, out_all, channels, T, T * N, N, sig.shape[1], hop, win, 1.0 / N,
                                                               True, st), 3))
            for F in args.frames:
                ctx = cf.fft_stft_stream_create(s, channels, hop, F, win, win, 1.0 / N, True, st)
                x, y = sig[:, :F * hop].contiguous(), torch.empty(channels, F * hop, device="cuda")
                spec = spec_all[:, :F].contiguous()
                ana = lambda: cf.fft_stft_stream_analyze(ctx, x, F * hop, F, spec, F * N, N, st)
                syn = lambda: cf.fft_stft_stream_synthesize(ctx, spec, F * N, N, F, y, F * hop, st)
                timed(ana, 10)
                timed(syn, 10)
                ta, ts = timed(ana, args.calls), timed(syn, args.calls)
                ma, ms = sum(ta) / len(ta), sum(ts) / len(ts)
                budget = F * hop / 48.0
                print(f"  {cfg:>9} {channels:5d} {F:3d} | {ma:10.4f} {max(ta):7.4f} {off_a:10.4f} {ma * T / F / off_a:6.2f} | {ms:9.4f} "
                      f"{max(ts):7.4f} {off_s:10.4f} {ms * T / F / off_s:6.2f} | {budget:9.3f} {budget / (ma + ms):8.1f}", flush=True)
                cf.fft_stft_stream_destroy(ctx)
                del x, y, spec
            del sig, spec_all, out_all
            torch.cuda.empty_cache()
        cf.fft_destroy_setup(s)


if __name__ == "__main__":
    main()
