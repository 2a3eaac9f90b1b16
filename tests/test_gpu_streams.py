"""Every device entry point on caller streams, from concurrent threads and inside CUDA graph capture.

include/chowdsp_fft_b200.h promises that a call on device pointers only enqueues work on the caller's `stream`, and
INTEGRATION.md §5 that a plan may be shared between threads.  A call that launched one kernel on stream 0, forgot to
join a helper lane of the L2-chunked multi-pass schedule back into the caller's stream, or kept per-thread state in a
process-wide object would still pass every test that calls with stream=None: the legacy default stream synchronises with
every blocking stream.  torch creates its streams non-blocking, so here:

1. Caller streams, late producer / early consumer.  On a fresh torch.cuda.Stream s every operand is NaN; s spins
   (torch.cuda._sleep), then copies the true inputs (windows, IRs, pre-loaded accumulators and delay lines too), the
   library call is made on s, every output is cloned on s right behind it and every input is overwritten with NaN.  The
   clone must equal the final output and, bit for bit, the same call made eagerly on the default stream, which must pass
   float64 (check_float64 of tests/test_gpu_routes.py) or the oracle's tolerance; the kernel reported is the dispatcher's
   (expected_kernel).  A few transforms also run with the special handles cudaStreamPerThread (2) and cudaStreamLegacy (1).
   The streaming convolver and STFT contexts run create (IR / windows produced late), process / synthesize and reset
   (while a call is still pending) on s.
2. Threads.  Six threads share the setups, each on its own stream with its own inputs, released together at a barrier
   (ctypes releases the GIL, so the calls overlap).  Each runs every case of part 1 twice in its own order, host-pointer
   calls (pageable staging, pinned zero-copy on cudaStreamPerThread, aligned_malloc churn, the drop-in calls) and its own
   convolver and STFT context block by block; every output must equal the serial default-stream result bit for bit.  A
   child process starts eight threads on a cold library: table builds, the first multi-pass call and the first host call
   race; then short-lived threads exit after a host call (their staging buffers are released on exit).  A targeted phase
   releases eight threads at a barrier straight into the L2-chunked schedule, round after round, half of them with late
   inputs: the helper lanes and fork / join events of that schedule must be the calling thread's own.
3. CUDA graphs.  Every stateless case is captured with torch.cuda.graph (capture_error_mode "global") after an eager
   warm-up and replayed three times on new inputs: each replay is bit-identical to an eager call and passes float64
   (launch_count() is checked not to move, a sanity check only: a replay never enters the library's host code, which is
   where launches are counted).  The stateful contexts keep their positions (the convolver's block
   count, the STFT frame counts) on the host, so a replayed capture would repeat one block: they are not replayable and
   are not captured here.
4. Two devices (skipped with fewer): a setup created on device 0 used from a thread bound to device 1, and one thread
   alternating multi-pass and host-pointer calls between the devices.

The last test checks that every route was reached on a caller stream, in threads and in capture.
"""
from __future__ import annotations

import json
import math
import os
import random
import subprocess
import sys
import threading

import numpy as np
import pytest

from tests.test_gpu_routes import Geometry, check_float64, data, expected_kernel, plain, unordered_perm
from tests.test_gpu_sizes import host_dft, widths

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SLEEP = 20_000_000          # cycles of torch.cuda._sleep in front of the late inputs
THREADS = 6
STREAM_PER_THREAD, STREAM_LEGACY = 2, 1
NAN = float("nan")

# routes of the cases below; test_every_route_was_reached checks each part reached all of them
ROUTES = ("fft_kernel", "pipe_kernel", "fft_kernel<13/14,32>", "wpipe_kernel", "fft_small_kernel", "mixq_kernel", "mixed_kernel",
          "tile_fft_kernel", "L2-chunked", "stft_forward", "wistft_kernel", "ristft_kernel", "istft_kernel", "juce", "juce mirror",
          "convolve", "accumulate", "pconv_kernel")
REACHED = {"stream": set(), "threads": set(), "graph": set()}
PARTS_RUN: set = set()


@pytest.fixture(scope="module")
def cf():
    import chowdsp_fft_b200 as m

    assert m.device_available(), "GPU tests need a CUDA device; there is no CPU fallback"
    return m


def bits(a) -> np.ndarray:
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def same_bits(a, b) -> bool:
    return a.shape == b.shape and np.array_equal(bits(a), bits(b))


def rel_l2(got, ref) -> float:
    d = np.asarray(got, np.float64) - np.asarray(ref, np.float64)
    return float(np.linalg.norm(d) / np.linalg.norm(np.asarray(ref, np.float64)))


def parity_tol(N: int) -> float:
    return 1e-6 * math.log2(N)


def hann(N: int) -> np.ndarray:
    return (0.5 - 0.5 * np.cos(2 * np.pi * np.arange(N) / N)).astype(np.float32)


# --------------------------------------------------------------------------------------------------
# cases: the operands, the call and the float64 / oracle check of one entry point
# --------------------------------------------------------------------------------------------------
class Setups:
    """Plans shared by every case, thread and seed (created before any thread starts)."""

    def __init__(self, cf):
        self.cf, self.plans = cf, {}

    def get(self, N: int, is_c: bool, avx: bool = True) -> int:
        k = (N, is_c, avx)
        if k not in self.plans:
            self.plans[k] = self.cf.fft_new_setup(N, self.cf.FFT_COMPLEX if is_c else self.cf.FFT_REAL, avx)
        return self.plans[k]

    def close(self):
        for s in self.plans.values():
            self.cf.fft_destroy_setup(s)
        self.plans.clear()


class Op:
    """One call of a stateless entry point.  `inputs`: operands the call reads (produced late), flat float32 arrays;
    `outputs`: operands it only writes, {name: float count} (NaN before the call); `results`: the operands compared
    afterwards (outputs and read-modify-write inputs); call(ptr, stream) makes the call on the operands' addresses;
    check(result) is the float64 / oracle check; kernel: prefix last_kernel() must report (None: not checked); notes: the
    call reports its kernel (the elementwise calls do not, so last_kernel() keeps the thread's previous one)."""

    def __init__(self, name, route, inputs, outputs, results, call, check, kernel=None, contains=None, notes=True):
        self.name, self.route, self.inputs, self.outputs, self.results = name, route, inputs, outputs, results
        self.call, self.check, self.kernel, self.contains, self.notes = call, check, kernel, contains, notes

    def same_kernel(self, got: str, want: str) -> None:
        if self.notes:
            assert got == want, (self.name, got, want)

    def check_kernel(self, got: str) -> None:
        if self.kernel is not None:
            assert got.startswith(self.kernel), (self.name, got, self.kernel)
        if self.contains is not None:
            assert self.contains in got, (self.name, got, self.contains)


def transform_op(name, N, is_c, ordered, backward, g: Geometry, route=None, contains=None):
    """fft_transform_batched (one-level) / fft_transform_strided (two-level) of one size, layout and geometry."""
    ws = widths(N, is_c)
    W = max(ws)
    avx = ws[W] if not ordered else True

    def make(cf, S, seed):
        setup = S.get(N, is_c, avx)
        nfl = 2 * N if is_c else N
        x, spec = data(N, is_c, g.batch, seed)
        perm = None if ordered else unordered_perm(N, is_c, W)
        rows = (spec if ordered else np.ascontiguousarray(spec[:, perm])) if backward else x
        ioff, ooff = g.rows("in"), g.rows("out")
        inp = np.full(int(ioff.max()) + nfl + 8, np.nan, np.float32)
        for r, o in enumerate(ioff):
            inp[o:o + nfl] = rows[r]  # overlapping frames: later rows rewrite the same samples
        out_len = int(ooff.max()) + nfl + 8
        frames = g.batch > 1 and len(set(ioff.tolist())) == g.batch and np.diff(np.sort(ioff)).min() < nfl
        direction = cf.FFT_BACKWARD if backward else cf.FFT_FORWARD

        def call(p, stream):
            if g.outer == 1:
                cf.fft_transform_batched(setup, p["in"] + 4 * g.in_off, p["out"] + 4 * g.out_off, g.inner, g.in_inner, g.out_inner,
                                         direction, ordered, stream)
            else:
                cf.fft_transform_strided(setup, p["in"] + 4 * g.in_off, p["out"] + 4 * g.out_off, g.outer, g.inner, g.in_outer,
                                         g.in_inner, g.out_outer, g.out_inner, direction, ordered, stream)

        def check(res):
            out = res["out"]
            mask = np.ones(out.shape[0], bool)
            for o in ooff:
                mask[o:o + nfl] = False
            assert np.isnan(out[mask]).all(), f"{name}: the transform wrote outside its rows"
            got = np.stack([out[o:o + nfl] for o in ooff])
            src = np.stack([inp[o:o + nfl] for o in ioff]) if frames else (spec if backward else x)
            ref = host_dft(src, N, is_c, backward)
            if not ordered and not backward:
                ref = ref[:, perm]
            check_float64(got, ref, N, is_c, ordered, backward, name)

        r, kernel = expected_kernel(N, is_c, backward, ordered, W, g)
        return Op(name, route or r, {"in": inp}, {"out": out_len}, ("out",), call, check, kernel, contains)

    return make


def stft_forward_op(N=2048, channels=3, frames=9, hop=512):
    """fft_stft_forward with a window that is produced late as well."""

    def make(cf, S, seed):
        setup = S.get(N, False)
        rng = np.random.default_rng(seed + 11)
        cs = (frames - 1) * hop + N + 6
        sig = rng.uniform(-1, 1, channels * cs).astype(np.float32)
        win = (hann(N) * rng.uniform(0.5, 1.5, N)).astype(np.float32)

        def call(p, stream):
            cf.fft_stft_forward(setup, p["sig"], p["spec"], channels, frames, cs, hop, frames * N, N, p["win"], True, stream)

        def check(res):
            s2 = sig.reshape(channels, cs)
            fr = np.stack([s2[:, f * hop:f * hop + N] for f in range(frames)], axis=1).reshape(-1, N).astype(np.float64)
            ref = host_dft(fr * win.astype(np.float64), N, False, False)
            got = res["spec"].reshape(-1, N)
            assert rel_l2(got, ref) < parity_tol(N), rel_l2(got, ref)

        return Op("stft_forward", "stft_forward", {"sig": sig, "win": win}, {"spec": channels * frames * N}, ("spec",), call, check)

    return make


def istft_op(name, N, hop, ordered, frames=7, channels=3):
    """fft_istft_overlap_add with a window produced late; every output sample is written."""
    from oracle import oracle as o

    W = o.simd_width(N, False)

    def make(cf, S, seed):
        setup = S.get(N, False)
        rng = np.random.default_rng(seed + 13)
        spec = rng.uniform(-1, 1, channels * frames * N).astype(np.float32)
        win = (hann(N) * rng.uniform(0.5, 1.5, N)).astype(np.float32)
        samples = (frames - 1) * hop + N
        cs = samples + 6

        def call(p, stream):
            cf.fft_istft_overlap_add(setup, p["spec"], p["sig"], channels, frames, frames * N, N, cs, hop, p["win"], 1.0 / N, ordered, stream)

        def check(res):
            got = res["sig"].reshape(channels, cs)
            want = o.np_istft_overlap_add(spec.reshape(channels, frames, N), N, hop, W, ordered, win, 1.0 / N)
            assert rel_l2(got[:, :samples], want) < parity_tol(N)
            assert np.isnan(got[:, samples:]).all()

        return Op(name, name, {"spec": spec, "win": win}, {"sig": channels * cs}, ("sig",), call, check, f"cfb::{name}<")

    return make


def juce_perform_op(inverse: bool, N=1024, batch=4):
    from oracle import oracle as o

    def make(cf, S, seed):
        setup = S.get(N, True)
        x = np.random.default_rng(seed + 17).uniform(-1, 1, batch * 2 * N).astype(np.float32)

        def call(p, stream):
            cf.fft_juce_perform_batched(setup, p["in"], p["out"], batch, 2 * N, 2 * N, inverse, stream)

        def check(res):
            want = o.np_juce_perform(x.reshape(batch, 2 * N), N, inverse)
            assert rel_l2(res["out"].reshape(batch, 2 * N), want) < parity_tol(N)

        # forward: the conventions coincide with fft_transform, so the plain transform kernel runs
        kernel = "cfb::fft_kernel_juce<" if inverse else expected_kernel(N, True, False, True, 8, plain(batch, 2 * N, 2 * N))[1]
        return Op(f"juce_perform_{'inv' if inverse else 'fwd'}", "juce", {"in": x}, {"out": batch * 2 * N}, ("out",), call, check, kernel)

    return make


def juce_real_forward_op(ignore: bool, N=1024, batch=4):
    """In place; with ignore_negative_freqs = 0 a second kernel writes the conjugate mirror."""
    from oracle import oracle as o

    def make(cf, S, seed):
        setup = S.get(N, False)
        buf = np.random.default_rng(seed + 19).uniform(-1, 1, batch * 2 * N).astype(np.float32)

        def call(p, stream):
            cf.fft_juce_real_forward_batched(setup, p["buf"], batch, 2 * N, ignore, stream)

        def check(res):
            got, want = res["buf"].reshape(batch, 2 * N), o.np_juce_real_forward(buf.reshape(batch, 2 * N), N, ignore)
            assert rel_l2(got[:, :N + 2], want[:, :N + 2]) < parity_tol(N)
            if ignore:
                assert same_bits(got[:, N + 2:], want[:, N + 2:])  # untouched
            else:
                assert rel_l2(got, want) < parity_tol(N)

        return Op(f"juce_real_forward_ignore{int(ignore)}", "juce" if ignore else "juce mirror", {"buf": buf}, {}, ("buf",), call, check,
                  "cfb::fft_kernel_juce<")

    return make


def juce_real_inverse_op(N=1024, batch=4):
    from oracle import oracle as o

    def make(cf, S, seed):
        setup = S.get(N, False)
        buf = np.random.default_rng(seed + 23).uniform(-1, 1, batch * 2 * N).astype(np.float32)

        def call(p, stream):
            cf.fft_juce_real_inverse_batched(setup, p["buf"], batch, 2 * N, stream)

        def check(res):
            got, want = res["buf"].reshape(batch, 2 * N), o.np_juce_real_inverse(buf.reshape(batch, 2 * N), N)
            assert rel_l2(got[:, :N], want[:, :N]) < parity_tol(N)

        return Op("juce_real_inverse", "juce", {"buf": buf}, {}, ("buf",), call, check, "cfb::fft_kernel_juce<")

    return make


def convolve_op(N=1024, batch=4):
    """ab += a b scaling on unordered spectra: ab is read too, so it is produced late."""
    from oracle import oracle as o

    W = o.simd_width(N, False)

    def make(cf, S, seed):
        setup = S.get(N, False)
        rng = np.random.default_rng(seed + 29)
        a, b, ab = (rng.uniform(-1, 1, batch * N).astype(np.float32) for _ in range(3))

        def call(p, stream):
            cf.fft_convolve_unordered_batched(setup, p["a"], p["b"], p["ab"], batch, N, N, N, 1.0 / N, stream)

        def check(res):
            want = o.np_convolve(a.reshape(batch, N), b.reshape(batch, N), ab.reshape(batch, N), N, False, W, 1.0 / N)
            assert rel_l2(res["ab"].reshape(batch, N), want) < 1e-6

        return Op("convolve_unordered", "convolve", {"a": a, "b": b, "ab": ab}, {}, ("ab",), call, check, notes=False)

    return make


def accumulate_op(n=4 * 1024):
    def make(cf, S, seed):
        setup = S.get(1024, False)
        rng = np.random.default_rng(seed + 31)
        a, b = (rng.uniform(-1, 1, n).astype(np.float32) for _ in range(2))

        def call(p, stream):
            cf.fft_accumulate_batched(setup, p["a"], p["b"], p["ab"], n, stream)

        def check(res):
            assert same_bits(res["ab"], a + b)

        return Op("accumulate", "accumulate", {"a": a, "b": b}, {"ab": n}, ("ab",), call, check, notes=False)

    return make


def pconv_op(N=256, channels=2, P=3, T=5):
    """T fft_partitioned_convolve_step calls in a row; the delay line carries the state between them."""
    from oracle import oracle as o

    W = o.simd_width(N, False)
    B = N // 2

    def make(cf, S, seed):
        setup = S.get(N, False)
        rng = np.random.default_rng(seed + 37)
        x = rng.uniform(-1, 1, (channels, T * B)).astype(np.float32)
        xpad = np.concatenate([np.zeros((channels, B), np.float32), x], axis=1)
        h = (rng.uniform(-1, 1, (channels, P, N)) / N).astype(np.float32)
        fdl = np.zeros(channels * P * N, np.float32)

        def call(p, stream):
            for t in range(T):
                cf.fft_partitioned_convolve_step(setup, p["win"] + 4 * t * B, xpad.shape[1], p["ir"], P * N, p["fdl"], P * N,
                                                 p["y"] + 4 * t * B, T * B, channels, P, t, 1.0 / N, stream)

        def check(res):
            want, _ = o.np_partitioned_convolve(x, h, N, P, W)
            assert rel_l2(res["y"].reshape(channels, T * B), want) < 1e-5

        return Op("partitioned_convolve_step", "pconv_kernel", {"win": xpad.ravel(), "ir": h.ravel(), "fdl": fdl}, {"y": channels * T * B},
                  ("y", "fdl"), call, check, "cfb::pconv_kernel<")

    return make


def three_pass_size(cf) -> int:
    """The smallest complex power of two whose plan has three passes (fft_large_factors l2 != 0)."""
    for e in range(15, 26):
        s = cf.fft_new_setup(1 << e, cf.FFT_COMPLEX)
        try:
            if cf.fft_large_factors(s)[1] != 0:
                return 1 << e
        finally:
            cf.fft_destroy_setup(s)
    raise AssertionError("no three-pass plan up to 2^25")


def make_ops(cf, sms: int, n3: int) -> list:
    """Every case of part 1, in table order."""
    def c(N):
        return 2 * N

    return [
        transform_op("c2c-4096", 4096, True, True, False, plain(5, c(4096), c(4096))),
        transform_op("c2c-8192-persistent", 8192, True, True, False, plain(2 * 2 * sms + 7, c(8192), c(8192))),
        transform_op("c2c-16384-persistent-bwd", 16384, True, False, True, plain(2 * sms + 7, c(16384), c(16384))),
        transform_op("c2c-16384-stride2mod4", 16384, True, True, False, plain(5, c(16384) + 2, c(16384) + 2)),
        transform_op("r2c-2048-unordered-4096", 2048, False, False, False, plain(4096, 2048, 2048)),
        transform_op("c2c-16-x1000", 16, True, True, False, plain(1000, c(16), c(16))),
        transform_op("c2c-768", 768, True, True, False, plain(5, c(768), c(768) + 4)),
        transform_op("c2c-400-bwd", 400, True, True, True, plain(5, c(400), c(400))),
        transform_op("c2c-2^17", 1 << 17, True, False, False, plain(3, c(1 << 17), c(1 << 17))),
        transform_op("real-2^18-bwd", 1 << 18, False, True, True, plain(3, 1 << 18, 1 << 18)),
        transform_op(f"c2c-{n3}-three-pass", n3, True, True, False, plain(2, c(n3), c(n3)), route="L2-chunked", contains="L2-chunked"),
        transform_op("strided-frames-2048", 2048, False, True, False, Geometry(2, 7, 6 * 2048 + 4, 2048 // 4, 7 * 2048, 2048)),
        transform_op("strided-two-level-1024", 1024, True, True, True,
                     Geometry(3, 5, 5 * (c(1024) + 4) + 12, c(1024) + 4, 5 * (c(1024) + 8) + 4, c(1024) + 8)),
        stft_forward_op(),
        istft_op("wistft_kernel", 2048, 512, True),
        istft_op("ristft_kernel", 4096, 1024, False),
        istft_op("istft_kernel", 512, 130, True),
        juce_perform_op(False),
        juce_perform_op(True),
        juce_real_forward_op(False),
        juce_real_forward_op(True),
        juce_real_inverse_op(),
        convolve_op(),
        accumulate_op(),
        pconv_op(),
    ]


# --------------------------------------------------------------------------------------------------
# running a case
# --------------------------------------------------------------------------------------------------
def upload(a: np.ndarray):
    return torch.from_numpy(a).cuda()


def eager(cf, op: Op):
    """The call on the default stream with stream=None, inputs in place before it: ({result: array}, last_kernel)."""
    bufs = {k: upload(v) for k, v in op.inputs.items()}
    bufs.update({k: torch.full((n,), NAN, device="cuda") for k, n in op.outputs.items()})
    torch.cuda.synchronize()
    op.call({k: t.data_ptr() for k, t in bufs.items()}, None)
    kernel = cf.last_kernel()
    torch.cuda.synchronize()
    return {k: bufs[k].cpu().numpy() for k in op.results}, kernel


def late(cf, op: Op, s):
    """Late producer / early consumer on stream s (torch.cuda.Stream, or an int handle whose stream is ordered with
    the legacy default stream).  Returns ({result: clone taken right behind the call}, last_kernel)."""
    on = s if not isinstance(s, int) else torch.cuda.default_stream()
    with torch.cuda.stream(on):
        src = {k: upload(v) for k, v in op.inputs.items()}
        bufs = {k: torch.full((v.size,), NAN, device="cuda") for k, v in op.inputs.items()}
        bufs.update({k: torch.full((n,), NAN, device="cuda") for k, n in op.outputs.items()})
    on.synchronize()
    with torch.cuda.stream(on):
        torch.cuda._sleep(SLEEP)
        for k in op.inputs:
            bufs[k].copy_(src[k])
        op.call({k: t.data_ptr() for k, t in bufs.items()}, s)
        kernel = cf.last_kernel()
        clones = {k: bufs[k].clone() for k in op.results}
        for k in op.inputs:
            bufs[k].fill_(NAN)
    on.synchronize()
    res = {k: t.cpu().numpy() for k, t in clones.items()}
    for k in op.results:
        if k not in op.inputs:
            assert same_bits(res[k], bufs[k].cpu().numpy()), f"{op.name}: {k} changed after the clone taken right behind the call"
    return res, kernel


def assert_same(op: Op, got: dict, want: dict, what: str) -> None:
    for k in op.results:
        a, b = got[k], want[k]
        if not same_bits(a, b):
            n = int((bits(a) != bits(b)).sum())
            raise AssertionError(f"{op.name} {what}: {k} differs from the eager default-stream call in {n} of {a.size} floats "
                                 f"({int(np.isnan(a).sum())} NaN)")


@pytest.fixture(scope="module")
def world(cf):
    """Shared setups, the cases and their eager default-stream results for seed 0."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    S = Setups(cf)
    n3 = three_pass_size(cf)
    makers = make_ops(cf, sms, n3)
    ops = [m(cf, S, 0) for m in makers]
    refs = []
    for op in ops:
        res, kernel = eager(cf, op)
        op.check_kernel(kernel)
        op.check(res)
        refs.append((res, kernel))
    yield dict(S=S, makers=makers, ops=ops, refs=refs, sms=sms, n3=n3)
    S.close()


# --------------------------------------------------------------------------------------------------
# 1. caller streams
# --------------------------------------------------------------------------------------------------
def test_late_producer_early_consumer_on_caller_streams(cf, world):
    """Every case on a fresh non-blocking stream with its inputs produced late and its outputs consumed early equals the
    eager default-stream call bit for bit (which passes float64), from the same kernel."""
    for op, (ref, kernel) in zip(world["ops"], world["refs"]):
        s = torch.cuda.Stream()
        got, k = late(cf, op, s)
        op.same_kernel(k, kernel)
        assert_same(op, got, ref, "on a caller stream")
        REACHED["stream"].add(op.route)
    PARTS_RUN.add("stream")


@pytest.mark.parametrize("handle", [STREAM_PER_THREAD, STREAM_LEGACY], ids=["cudaStreamPerThread", "cudaStreamLegacy"])
def test_special_stream_handles(cf, world, handle):
    """cudaStreamPerThread and cudaStreamLegacy passed as `stream`: a single-kernel route and the L2-chunked route, with
    inputs produced late on the legacy default stream and outputs consumed early there."""
    picks = [i for i, op in enumerate(world["ops"]) if op.name in ("c2c-4096", "strided-frames-2048") or op.route == "L2-chunked"]
    assert len(picks) == 3
    for i in picks:
        op, (ref, kernel) = world["ops"][i], world["refs"][i]
        got, k = late(cf, op, handle)
        op.same_kernel(k, kernel)
        assert_same(op, got, ref, f"on stream handle {handle}")


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x, np.float32)).cuda()


def linear(x, h):
    """y_c = x_c * h_c in float64, first x.shape[1] samples (as tests/test_gpu_convolver.py)."""
    n = x.shape[1] + h.shape[1] - 1
    size = 1 << (n - 1).bit_length()
    y = np.fft.irfft(np.fft.rfft(x.astype(np.float64), size) * np.fft.rfft(h.astype(np.float64), size), size)
    return y[:, :x.shape[1]]


class ConvolverRun:
    """One convolver context: create with the IR, blocks of input, reset, the same blocks again."""
    B, L, CH, T = 64, 1000, 2, 24

    def __init__(self, seed):
        rng = np.random.default_rng(seed + 41)
        self.h = (rng.uniform(-1, 1, (self.CH, self.L)) / np.sqrt(self.L)).astype(np.float32)
        self.x = rng.uniform(-1, 1, (self.CH, self.T * self.B)).astype(np.float32)
        self.junk = rng.uniform(-1, 1, (self.CH, self.B)).astype(np.float32)

    def create(self, cf, s=None):
        """With a stream: the IR is produced late on it and overwritten with NaN once create returns."""
        if s is None:
            return cf.fft_convolver_create(self.CH, self.B, dev(self.h), self.L, self.L)
        src, ir = dev(self.h), torch.full((self.CH, self.L), NAN, device="cuda")
        torch.cuda.synchronize()
        with torch.cuda.stream(s):
            torch.cuda._sleep(SLEEP)
            ir.copy_(src)
            ctx = cf.fft_convolver_create(self.CH, self.B, ir, self.L, self.L, s)
            ir.fill_(NAN)
        s.synchronize()
        return ctx

    def blocks(self, cf, ctx, s=None, late_input=True):
        """All T blocks; with a stream, each block's input is produced late and overwritten after the call."""
        B, T = self.B, self.T
        y = torch.full((self.CH, T * B), NAN, device="cuda")
        xin = torch.full((self.CH, B), NAN, device="cuda")
        src = dev(self.x)
        torch.cuda.synchronize()
        with torch.cuda.stream(s if s is not None else torch.cuda.current_stream()):
            for t in range(T):
                if s is not None and late_input:
                    torch.cuda._sleep(SLEEP // 8)
                xin.copy_(src[:, t * B:(t + 1) * B])
                cf.fft_convolver_process(ctx, xin, B, y.data_ptr() + 4 * t * B, T * B, s)
                if s is not None:
                    xin.fill_(NAN)
        (s or torch.cuda.current_stream()).synchronize()
        return y.cpu().numpy()

    def reset_pending(self, cf, ctx, s=None):
        """A process call still pending on the stream (behind a spin), then reset on the same stream."""
        junk = dev(self.junk)
        yj = torch.empty((self.CH, self.B), device="cuda")
        torch.cuda.synchronize()
        with torch.cuda.stream(s if s is not None else torch.cuda.current_stream()):
            if s is not None:
                torch.cuda._sleep(SLEEP)
            cf.fft_convolver_process(ctx, junk, self.B, yj, self.B, s)
            cf.fft_convolver_reset(ctx, s)
        (s or torch.cuda.current_stream()).synchronize()


def test_convolver_on_a_caller_stream(cf):
    """create (IR produced late), process (input produced late), reset behind a pending process, process again, all on a
    non-blocking stream: the same bits as the context run on the default stream, and the float64 linear convolution."""
    run = ConvolverRun(0)
    ref_ctx = run.create(cf)
    s = torch.cuda.Stream()
    ctx = run.create(cf, s)
    try:
        want = run.blocks(cf, ref_ctx)
        got = run.blocks(cf, ctx, s)
        assert same_bits(got, want), "convolver on a caller stream differs from the default-stream context"
        assert rel_l2(got, linear(run.x, run.h)) < 1e-5
        run.reset_pending(cf, ctx, s)
        again = run.blocks(cf, ctx, s)
        assert same_bits(again, want), "reset behind a pending process call did not return the context to silence"
    finally:
        cf.fft_convolver_destroy(ctx)
        cf.fft_convolver_destroy(ref_ctx)


class StftRun:
    """One streaming STFT context: create with both windows, analyze and synthesize block by block, reset, again."""
    N, HOP, CH, MAXF, J = 1024, 256, 2, 4, 14

    def __init__(self, seed):
        rng = np.random.default_rng(seed + 43)
        N = self.N
        self.aw = (hann(N) * rng.uniform(0.5, 1.5, N)).astype(np.float32)
        self.sw = (hann(N) * rng.uniform(0.5, 1.5, N)).astype(np.float32)
        self.x = rng.uniform(-1, 1, (self.CH, self.J * self.HOP)).astype(np.float32)
        self.spec = rng.uniform(-1, 1, (self.CH, self.J, N)).astype(np.float32)
        self.split = [1, 3, 4, 2, 4]
        assert sum(self.split) == self.J

    def create(self, cf, setup, s=None):
        if s is None:
            return cf.fft_stft_stream_create(setup, self.CH, self.HOP, self.MAXF, dev(self.aw), dev(self.sw), 1.0 / self.N, True)
        srcs = [dev(self.aw), dev(self.sw)]
        wins = [torch.full((self.N,), NAN, device="cuda") for _ in range(2)]
        torch.cuda.synchronize()
        with torch.cuda.stream(s):
            torch.cuda._sleep(SLEEP)
            for w, src in zip(wins, srcs):
                w.copy_(src)
            ctx = cf.fft_stft_stream_create(setup, self.CH, self.HOP, self.MAXF, wins[0], wins[1], 1.0 / self.N, True, s)
            for w in wins:
                w.fill_(NAN)
        s.synchronize()
        return ctx

    def blocks(self, cf, ctx, s=None):
        """(spectra of analyze, signal of synthesize); with a stream, each call's input is produced late."""
        N, hop, J, CH = self.N, self.HOP, self.J, self.CH
        spec_out = torch.full((CH, J, N), NAN, device="cuda")
        y = torch.full((CH, J * hop), NAN, device="cuda")
        xin = torch.full((CH, self.MAXF * hop), NAN, device="cuda")
        sin = torch.full((CH, self.MAXF, N), NAN, device="cuda")
        xs, ss = dev(self.x), dev(self.spec)
        torch.cuda.synchronize()
        stream = s if s is not None else torch.cuda.current_stream()
        with torch.cuda.stream(stream):
            f = 0
            for n in self.split:
                if s is not None:
                    torch.cuda._sleep(SLEEP // 8)
                xin[:, :n * hop].copy_(xs[:, f * hop:(f + n) * hop])
                sin[:, :n].copy_(ss[:, f:f + n])
                cf.fft_stft_stream_analyze(ctx, xin, self.MAXF * hop, n, spec_out.data_ptr() + 4 * f * N, J * N, N, s)
                cf.fft_stft_stream_synthesize(ctx, sin, self.MAXF * N, N, n, y.data_ptr() + 4 * f * hop, J * hop, s)
                if s is not None:
                    xin.fill_(NAN)
                    sin.fill_(NAN)
                f += n
        stream.synchronize()
        return spec_out.cpu().numpy(), y.cpu().numpy()

    def reset_pending(self, cf, ctx, s=None):
        hop, N = self.HOP, self.N
        xin, sp = torch.rand((self.CH, hop), device="cuda"), torch.rand((self.CH, 1, N), device="cuda")
        so, yo = torch.empty((self.CH, 1, N), device="cuda"), torch.empty((self.CH, hop), device="cuda")
        torch.cuda.synchronize()
        stream = s if s is not None else torch.cuda.current_stream()
        with torch.cuda.stream(stream):
            if s is not None:
                torch.cuda._sleep(SLEEP)
            cf.fft_stft_stream_analyze(ctx, xin, hop, 1, so, N, N, s)
            cf.fft_stft_stream_synthesize(ctx, sp, N, N, 1, yo, hop, s)
            cf.fft_stft_stream_reset(ctx, s)
        stream.synchronize()


def test_stft_stream_on_a_caller_stream(cf):
    """create (both windows produced late), analyze and synthesize (inputs produced late), reset behind pending calls, again,
    on a non-blocking stream: the bits of the default-stream context; synthesis within the oracle's tolerance."""
    from oracle import oracle as o

    run = StftRun(0)
    setup = cf.fft_new_setup(run.N, cf.FFT_REAL)
    ref_ctx = run.create(cf, setup)
    s = torch.cuda.Stream()
    ctx = run.create(cf, setup, s)
    try:
        want = run.blocks(cf, ref_ctx)
        got = run.blocks(cf, ctx, s)
        assert same_bits(got[0], want[0]) and same_bits(got[1], want[1]), "STFT context on a caller stream differs"
        ola = o.np_istft_overlap_add(run.spec, run.N, run.HOP, 8, True, run.sw, 1.0 / run.N)[:, :run.J * run.HOP]
        assert rel_l2(got[1], ola) < parity_tol(run.N)
        run.reset_pending(cf, ctx, s)
        again = run.blocks(cf, ctx, s)
        assert same_bits(again[0], want[0]) and same_bits(again[1], want[1]), "reset behind pending calls did not return to silence"
    finally:
        cf.fft_stft_stream_destroy(ctx)
        cf.fft_stft_stream_destroy(ref_ctx)
        cf.fft_destroy_setup(setup)


# --------------------------------------------------------------------------------------------------
# 2. threads sharing setups
# --------------------------------------------------------------------------------------------------
HOST_N = 1024


def host_tasks(cf, setup, real_setup, seed):
    """Host-pointer calls of one thread: [(name, fn() -> array)]; device-pointer references come from host_refs."""
    rng = np.random.default_rng(seed + 47)
    nfl = 2 * HOST_N
    x = rng.uniform(-1, 1, (8, nfl)).astype(np.float32)
    a, b, ab = (rng.uniform(-1, 1, HOST_N).astype(np.float32) for _ in range(3))

    def pageable():
        out = np.full_like(x, NAN)
        cf.fft_transform_batched(setup, x, out, 8, nfl, nfl, cf.FFT_FORWARD, True)
        return out

    def pinned():  # 8 x 8 KiB: under the zero-copy limit, so the kernel reads the mapped buffers on cudaStreamPerThread
        hin, hout = cf.aligned_array(8 * nfl), cf.aligned_array(8 * nfl)
        try:
            hin[:] = x.ravel()
            hout[:] = NAN
            cf.fft_transform_batched(setup, hin, hout, 8, nfl, nfl, cf.FFT_FORWARD, True)
            return hout.copy().reshape(8, nfl)
        finally:
            cf.aligned_free(hin.ctypes.data)
            cf.aligned_free(hout.ctypes.data)

    def churn():  # allocations and frees between calls bump the classify cache generation
        out = None
        for k in range(3):
            extra = cf.aligned_array(1024 * (k + 1))
            hin, hout = cf.aligned_array(nfl), cf.aligned_array(nfl)
            try:
                hin[:] = x[k]
                cf.fft_transform(setup, hin, hout, None, cf.FFT_FORWARD)
                row = hout.copy()
            finally:
                cf.aligned_free(extra.ctypes.data)
                cf.aligned_free(hin.ctypes.data)
                cf.aligned_free(hout.ctypes.data)
            out = row[None] if out is None else np.concatenate([out, row[None]])
        return out

    def dropin():
        out = np.full(nfl, NAN, np.float32)
        cf.fft_transform(setup, np.ascontiguousarray(x[3]), out, None, cf.FFT_FORWARD)
        return out[None]

    def dropin_convolve():
        acc = ab.copy()
        cf.fft_convolve_unordered(real_setup, a, b, acc, 1.0 / HOST_N)
        return acc[None]

    return [("pageable", pageable), ("pinned", pinned), ("churn", churn), ("dropin", dropin), ("dropin_convolve", dropin_convolve)], (x, a, b, ab)


def host_refs(cf, setup, real_setup, operands) -> dict:
    """The device-pointer results the host tasks must reproduce."""
    x, a, b, ab = operands
    nfl = 2 * HOST_N
    dx, dy = dev(x), torch.full((8, nfl), NAN, device="cuda")
    cf.fft_transform_batched(setup, dx, dy, 8, nfl, nfl, cf.FFT_FORWARD, True)
    acc = dev(ab)
    cf.fft_convolve_unordered_batched(real_setup, dev(a), dev(b), acc, 1, HOST_N, HOST_N, HOST_N, 1.0 / HOST_N)
    torch.cuda.synchronize()
    y = dy.cpu().numpy()
    return {"pageable": y, "pinned": y, "churn": y[:3], "dropin": y[3:4], "dropin_convolve": acc.cpu().numpy()[None]}


def test_threads_share_setups_on_their_own_streams(cf, world):
    """Six threads, released together, each on its own stream with its own inputs: every case of part 1 twice in a per-thread
    order, host-pointer calls, and a convolver and an STFT context of their own block by block; every result equals the
    serial default-stream result bit for bit and every thread sees its own last_kernel()."""
    S, makers = world["S"], world["makers"]
    setup_c, setup_r = S.get(HOST_N, True), S.get(HOST_N, False)
    stft_setup = S.get(StftRun.N, False)
    plans = []
    for t in range(THREADS):
        seed = 1000 * (t + 1)
        ops = [m(cf, S, seed) for m in makers]
        refs = [eager(cf, op) for op in ops]
        tasks, operands = host_tasks(cf, setup_c, setup_r, seed)
        conv, stft = ConvolverRun(seed), StftRun(seed)
        conv_ref_ctx, stft_ref_ctx = conv.create(cf), stft.create(cf, stft_setup)
        conv_want, stft_want = conv.blocks(cf, conv_ref_ctx), stft.blocks(cf, stft_ref_ctx)
        cf.fft_convolver_destroy(conv_ref_ctx)
        cf.fft_stft_stream_destroy(stft_ref_ctx)
        plans.append(dict(seed=seed, ops=ops, refs=refs, tasks=tasks, host_refs=host_refs(cf, setup_c, setup_r, operands),
                          conv=conv, conv_ctx=conv.create(cf), conv_want=conv_want,
                          stft=stft, stft_ctx=stft.create(cf, stft_setup), stft_want=stft_want))
    torch.cuda.synchronize()
    barrier = threading.Barrier(THREADS)
    errors, reached = [], set()
    lock = threading.Lock()

    def worker(plan):
        try:
            s = torch.cuda.Stream()
            rnd = random.Random(plan["seed"])
            order = [("op", i) for i in range(len(plan["ops"]))] * 2 + [("host", i) for i in range(len(plan["tasks"]))] * 2
            rnd.shuffle(order)
            conv, stft = plan["conv"], plan["stft"]
            conv_y = torch.full((conv.CH, conv.T * conv.B), NAN, device="cuda")
            conv_x = dev(conv.x)
            stft_spec = torch.full((stft.CH, stft.J, stft.N), NAN, device="cuda")
            stft_y = torch.full((stft.CH, stft.J * stft.HOP), NAN, device="cuda")
            stft_x, stft_s = dev(stft.x), dev(stft.spec)
            torch.cuda.synchronize()
            conv_t, stft_k, stft_f = 0, 0, 0
            barrier.wait()
            for kind, i in order:
                if kind == "op":
                    op, (ref, kernel) = plan["ops"][i], plan["refs"][i]
                    got, k = late(cf, op, s)
                    op.same_kernel(k, kernel)
                    assert_same(op, got, ref, f"in thread seed {plan['seed']}")
                    with lock:
                        reached.add(op.route)
                else:
                    name, fn = plan["tasks"][i]
                    out = fn()
                    assert same_bits(out, plan["host_refs"][name]), f"host path {name} in thread seed {plan['seed']}"
                # the thread's contexts advance one block between the other calls, on the thread's stream
                B = conv.B
                if conv_t < conv.T:
                    cf.fft_convolver_process(plan["conv_ctx"], conv_x.data_ptr() + 4 * conv_t * B, conv.T * B,
                                             conv_y.data_ptr() + 4 * conv_t * B, conv.T * B, s)
                    conv_t += 1
                if stft_k < len(stft.split):
                    n, f, hop, N = stft.split[stft_k], stft_f, stft.HOP, stft.N
                    cf.fft_stft_stream_analyze(plan["stft_ctx"], stft_x.data_ptr() + 4 * f * hop, stft.J * hop, n,
                                               stft_spec.data_ptr() + 4 * f * N, stft.J * N, N, s)
                    cf.fft_stft_stream_synthesize(plan["stft_ctx"], stft_s.data_ptr() + 4 * f * N, stft.J * N, N, n,
                                                  stft_y.data_ptr() + 4 * f * hop, stft.J * hop, s)
                    stft_k, stft_f = stft_k + 1, f + n
            assert conv_t == conv.T and stft_k == len(stft.split)
            s.synchronize()
            assert same_bits(conv_y.cpu().numpy(), plan["conv_want"]), f"convolver in thread seed {plan['seed']}"
            assert same_bits(stft_spec.cpu().numpy(), plan["stft_want"][0]), f"STFT analysis in thread seed {plan['seed']}"
            assert same_bits(stft_y.cpu().numpy(), plan["stft_want"][1]), f"STFT synthesis in thread seed {plan['seed']}"
        except BaseException as e:  # noqa: BLE001 -- reported by the main thread
            barrier.abort()
            with lock:
                errors.append(f"{type(e).__name__}: {e}")

    threads = [threading.Thread(target=worker, args=(p,)) for p in plans]
    try:
        for th in threads:
            th.start()
        for th in threads:
            th.join(timeout=600)
        assert not any(th.is_alive() for th in threads), "a worker thread did not finish"
    finally:
        torch.cuda.synchronize()
        for p in plans:
            cf.fft_convolver_destroy(p["conv_ctx"])
            cf.fft_stft_stream_destroy(p["stft_ctx"])
    assert not errors, errors[:4]
    REACHED["threads"] |= reached
    PARTS_RUN.add("threads")


RACE_THREADS, RACE_ROUNDS = 8, 12


def test_threads_race_into_the_l2_chunked_schedule(cf, world):
    """Eight threads enter the L2-chunked three-pass schedule together, round after round, each on its own stream.  A
    schedule run records a fork event on the caller's stream and makes each helper lane wait on it at the lane's first
    use, so the lanes and events must belong to the calling thread.  Even threads produce their inputs late (behind a
    spin), odd threads have them ready: a late thread whose lanes waited on an early thread's fork would run its chunks
    on NaN inputs.  1 MiB chunks on 4 lanes give every call many chunks and lane first-uses.  Every result equals the
    serial result bit for bit, which passes float64."""
    i = next(i for i, op in enumerate(world["ops"]) if op.route == "L2-chunked")
    make = world["makers"][i]
    cf.set_tuning("l2_chunk_mb", 1)
    cf.set_tuning("l2_lanes", 4)
    try:
        ops = [make(cf, world["S"], 9000 + t) for t in range(RACE_THREADS)]
        refs = []
        for op in ops:
            res, kernel = eager(cf, op)
            op.check_kernel(kernel)
            op.check(res)
            refs.append(res)
        # per thread: its stream, the true inputs on the device and the operands the call uses, allocated on that stream
        streams = [torch.cuda.Stream() for _ in ops]
        state = []
        for op, s in zip(ops, streams):
            with torch.cuda.stream(s):
                src = {k: upload(v) for k, v in op.inputs.items()}
                bufs = {k: torch.full((v.size,), NAN, device="cuda") for k, v in op.inputs.items()}
                bufs.update({k: torch.full((n,), NAN, device="cuda") for k, n in op.outputs.items()})
            state.append((src, bufs, {k: t.data_ptr() for k, t in bufs.items()}))
        torch.cuda.synchronize()
        barrier = threading.Barrier(RACE_THREADS)
        errors, lock = [], threading.Lock()

        def worker(t):
            op, s, (src, bufs, ptrs) = ops[t], streams[t], state[t]
            produce_late = t % 2 == 0
            try:
                for r in range(RACE_ROUNDS):
                    with torch.cuda.stream(s):
                        for k in bufs:
                            bufs[k].fill_(NAN)
                        if not produce_late:
                            for k in op.inputs:
                                bufs[k].copy_(src[k])
                    s.synchronize()
                    barrier.wait()
                    with torch.cuda.stream(s):
                        if produce_late:
                            torch.cuda._sleep(SLEEP)
                            for k in op.inputs:
                                bufs[k].copy_(src[k])
                        op.call(ptrs, s)
                        clones = {k: bufs[k].clone() for k in op.results}
                        for k in op.inputs:
                            bufs[k].fill_(NAN)
                    s.synchronize()
                    assert "L2-chunked" in cf.last_kernel(), cf.last_kernel()
                    assert_same(op, {k: c.cpu().numpy() for k, c in clones.items()}, refs[t], f"thread {t} round {r}")
            except BaseException as e:  # noqa: BLE001 -- reported by the main thread
                barrier.abort()
                with lock:
                    errors.append(f"{type(e).__name__}: {e}")

        threads = [threading.Thread(target=worker, args=(t,)) for t in range(RACE_THREADS)]
        for th in threads:
            th.start()
        for th in threads:
            th.join(timeout=600)
        assert not any(th.is_alive() for th in threads), "a worker thread did not finish"
        assert not errors, errors[:4]
    finally:
        torch.cuda.synchronize()
        cf.set_tuning("l2_chunk_mb", -1)
        cf.set_tuning("l2_lanes", -1)


COLD_START = r"""
import json, sys, threading
import numpy as np, torch
import chowdsp_fft_b200 as cf
from tests.test_gpu_routes import check_float64
from tests.test_gpu_sizes import host_dft

torch.cuda.set_device(0)
THREADS, SIZES = 8, [(2048, True), (4096, False), (768, True), (1 << 21, True)]
barrier, lock, errors, kernels = threading.Barrier(THREADS), threading.Lock(), [], set()

def rows(N, is_c, batch, seed):
    return np.random.default_rng(seed).uniform(-1, 1, (batch, 2 * N if is_c else N)).astype(np.float32)

def worker(t):
    try:
        barrier.wait()
        plans = {(N, c): cf.fft_new_setup(N, cf.FFT_COMPLEX if c else cf.FFT_REAL) for N, c in SIZES}  # tables race under the mutex
        s = torch.cuda.Stream()
        for (N, c), p in plans.items():
            batch = 1 if N > 4096 else 5
            x = rows(N, c, batch, 100 * t + N)
            if N <= 4096:  # the thread's first host-pointer call: its staging streams and buffers
                out = np.full_like(x, np.nan)
                cf.fft_transform_batched(p, x, out, batch, x.shape[1], x.shape[1], cf.FFT_FORWARD, True)
                check_float64(out, host_dft(x, N, c, False), N, c, True, False, f"host N={N} thread {t}")
            with torch.cuda.stream(s):  # the thread's first multi-pass call: its helper lanes and events
                dx = torch.from_numpy(x).cuda()
                dy = torch.full_like(dx, float("nan"))
                cf.fft_transform_batched(p, dx, dy, batch, x.shape[1], x.shape[1], cf.FFT_FORWARD, True, s)
                k = cf.last_kernel()
            s.synchronize()
            check_float64(dy.cpu().numpy(), host_dft(x, N, c, False), N, c, True, False, f"device N={N} thread {t}")
            with lock:
                kernels.add(k.split(" ")[0] + (" L2-chunked" if "L2-chunked" in k else ""))
        for p in plans.values():
            cf.fft_destroy_setup(p)
    except BaseException as e:
        barrier.abort()
        with lock:
            errors.append(f"thread {t}: {type(e).__name__}: {e}")

ths = [threading.Thread(target=worker, args=(t,)) for t in range(THREADS)]
for th in ths: th.start()
for th in ths: th.join()

# short-lived threads: one host call each, then exit (the thread's staging streams and buffers are released)
p = cf.fft_new_setup(1024, cf.FFT_COMPLEX)
x = rows(1024, True, 3, 7)
def short(t):
    try:
        out = np.full_like(x, np.nan)
        cf.fft_transform_batched(p, x, out, 3, 2048, 2048, cf.FFT_FORWARD, True)
        check_float64(out, host_dft(x, 1024, True, False), 1024, True, True, False, f"short-lived thread {t}")
    except BaseException as e:
        with lock:
            errors.append(f"short-lived thread {t}: {type(e).__name__}: {e}")
for t in range(16):
    th = threading.Thread(target=short, args=(t,)); th.start(); th.join()
out = np.full_like(x, np.nan)
cf.fft_transform_batched(p, x, out, 3, 2048, 2048, cf.FFT_FORWARD, True)
check_float64(out, host_dft(x, 1024, True, False), 1024, True, True, False, "main thread after the short-lived threads")
cf.fft_destroy_setup(p)
torch.cuda.synchronize()
print(json.dumps({"errors": errors, "kernels": sorted(kernels)}))
sys.exit(1 if errors else 0)
"""


def test_cold_start_threads_in_a_child_process(cf):
    """Eight threads on a library that has built nothing yet: the same sizes' tables, the first multi-pass call (helper
    lanes) and the first host call (staging) race; then sixteen short-lived threads make a host call each and exit, and
    the main thread's next call is still right.  Every result passes float64."""
    env = dict(os.environ, PYTHONNOUSERSITE="1")
    r = subprocess.run([sys.executable, "-c", COLD_START], capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    log = r.stdout[-4000:] + "\n" + r.stderr[-4000:]
    assert r.returncode == 0, log
    summary = json.loads(r.stdout.strip().splitlines()[-1])
    assert not summary["errors"], summary
    assert any("L2-chunked" in k for k in summary["kernels"]), summary


# --------------------------------------------------------------------------------------------------
# 3. CUDA graph capture
# --------------------------------------------------------------------------------------------------
def test_graph_capture_and_replay(cf, world):
    """Every stateless case captured after an eager warm-up (torch.cuda.graph, capture_error_mode "global") and replayed on
    three new inputs: each replay is bit-identical to an eager call on that input and passes float64.  launch_count() must
    not move across a replay; that is a sanity check only (replays never enter the library's host code, where launches are
    counted), not a proof of anything."""
    S = world["S"]
    for m, op in zip(world["makers"], world["ops"]):
        bufs = {k: upload(v) for k, v in op.inputs.items()}
        bufs.update({k: torch.full((n,), NAN, device="cuda") for k, n in op.outputs.items()})
        ptrs = {k: t.data_ptr() for k, t in bufs.items()}
        torch.cuda.synchronize()
        op.call(ptrs, None)  # warm-up
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            op.call(ptrs, torch.cuda.current_stream().cuda_stream)
            kernel = cf.last_kernel()
        op.check_kernel(kernel)
        for r in range(3):
            new = m(cf, S, 7000 + r)
            for k, v in new.inputs.items():
                bufs[k].copy_(torch.from_numpy(v))
            for k in new.outputs:
                bufs[k].fill_(NAN)
            torch.cuda.synchronize()
            n0 = cf.launch_count()
            g.replay()
            torch.cuda.synchronize()
            assert cf.launch_count() == n0, f"{op.name}: launch count moved across a replay"
            got = {k: bufs[k].cpu().numpy() for k in new.results}
            want, _ = eager(cf, new)
            assert_same(new, got, want, f"replay {r}")
            new.check(got)
        del g
        REACHED["graph"].add(op.route)
    PARTS_RUN.add("graph")


def test_graph_capture_without_warm_up_on_a_fresh_thread(cf, world):
    """Every stateless case captured on a thread that has made no library call before, with no eager warm-up, and replayed
    on a new input: bit-identical to an eager call, and within float64.  The multi-pass cases used to fail here: their
    first call on a thread set the device pool's release threshold, which invalidated the capture; setup now sets it."""
    S, errors = world["S"], []

    def capture(m, op):
        try:
            bufs = {k: upload(v) for k, v in op.inputs.items()}
            bufs.update({k: torch.full((n,), NAN, device="cuda") for k, n in op.outputs.items()})
            ptrs = {k: t.data_ptr() for k, t in bufs.items()}
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                op.call(ptrs, torch.cuda.current_stream().cuda_stream)
            new = m(cf, S, 8000)
            for k, v in new.inputs.items():
                bufs[k].copy_(torch.from_numpy(v))
            for k in new.outputs:
                bufs[k].fill_(NAN)
            torch.cuda.synchronize()
            g.replay()
            torch.cuda.synchronize()
            got = {k: bufs[k].cpu().numpy() for k in new.results}
            want, _ = eager(cf, new)
            assert_same(new, got, want, "replay of a capture without warm-up")
            new.check(got)
        except BaseException as e:  # noqa: BLE001 -- reported by the main thread
            errors.append(f"{op.name}: {type(e).__name__}: {str(e)[:300]}")

    for m, op in zip(world["makers"], world["ops"]):
        th = threading.Thread(target=capture, args=(m, op))
        th.start()
        th.join(timeout=300)
        assert not th.is_alive(), op.name
    assert not errors, errors


# --------------------------------------------------------------------------------------------------
# 4. two devices
# --------------------------------------------------------------------------------------------------
def two_devices():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")


def device_call(cf, setup, N, is_c, x, device, stream=None):
    with torch.cuda.device(device):
        dx = torch.from_numpy(x).to(f"cuda:{device}")
        dy = torch.full_like(dx, NAN)
        cf.fft_transform_batched(setup, dx, dy, x.shape[0], x.shape[1], x.shape[1], cf.FFT_FORWARD, True, stream)
        torch.cuda.synchronize(device)
        return dy.cpu().numpy()


def in_thread(fn):
    errors = []

    def run():
        try:
            fn()
        except BaseException as e:  # noqa: BLE001
            errors.append(f"{type(e).__name__}: {e}")

    th = threading.Thread(target=run)
    th.start()
    th.join(timeout=600)
    assert not th.is_alive() and not errors, errors


def test_setup_from_device_0_used_on_device_1(cf):
    """A setup created on device 0, used from a thread bound to device 1: its tables are built there on first use."""
    two_devices()
    torch.cuda.set_device(0)
    cases = [(4096, True), (2048, False), (768, True)]
    plans = {c: cf.fft_new_setup(c[0], cf.FFT_COMPLEX if c[1] else cf.FFT_REAL) for c in cases}

    def body():
        torch.cuda.set_device(1)
        s = torch.cuda.Stream(device=1)
        for (N, is_c), p in plans.items():
            x = data(N, is_c, 5, N)[0]
            got = device_call(cf, p, N, is_c, x, 1, s)
            check_float64(got, host_dft(x, N, is_c, False), N, is_c, True, False, f"N={N} on device 1")

    try:
        in_thread(body)
    finally:
        for p in plans.values():
            cf.fft_destroy_setup(p)


def test_one_thread_alternates_devices(cf, world):
    """One thread alternates multi-pass (L2-chunked) and host-pointer calls between the devices: the helper lanes and the
    staging buffers are rebuilt for each device."""
    two_devices()
    n3 = world["n3"]
    torch.cuda.set_device(0)
    big = cf.fft_new_setup(n3, cf.FFT_COMPLEX)
    small = cf.fft_new_setup(1024, cf.FFT_COMPLEX)

    def body():
        xb = data(n3, True, 1, 5)[0]
        xs = data(1024, True, 3, 6)[0]
        refb, refs = host_dft(xb, n3, True, False), host_dft(xs, 1024, True, False)
        for rnd in range(2):
            for d in (0, 1, 0, 1):
                torch.cuda.set_device(d)
                got = device_call(cf, big, n3, True, xb, d, torch.cuda.Stream(device=d))
                assert "L2-chunked" in cf.last_kernel()
                check_float64(got, refb, n3, True, True, False, f"multi-pass on device {d}")
                out = np.full_like(xs, NAN)
                cf.fft_transform_batched(small, xs, out, 3, 2048, 2048, cf.FFT_FORWARD, True)
                check_float64(out, refs, 1024, True, True, False, f"host call on device {d}")

    try:
        in_thread(body)
    finally:
        torch.cuda.set_device(0)
        cf.fft_destroy_setup(big)
        cf.fft_destroy_setup(small)


# --------------------------------------------------------------------------------------------------
def test_every_route_was_reached():
    """Every route was reached on a caller stream, in threads and in capture (run with the whole module)."""
    if PARTS_RUN != {"stream", "threads", "graph"}:
        pytest.skip("only part of the module ran")
    missing = {part: [r for r in ROUTES if r not in got] for part, got in REACHED.items()}
    assert not any(missing.values()), f"routes never reached: {missing}"
