"""Replacing the IR of a live streaming convolver (fft_convolver_set_ir) on the GPU: an instant swap is bit-identical to a
fresh context built with the new IR from the swap on, across the schedule's boundaries and firing phases; a crossfade
matches the float64 mix of both convolutions and is bit-identical to the fresh context once over; repeated swaps, reset
during a fade, the unchanged hot path and memory, stream ordering, argument errors, and one case under compute-sanitizer."""
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

from tests.test_gpu_convolver import BMAX, linear

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def cf():
    import chowdsp_fft_b200 as m

    assert m.device_available(), "GPU tests need a CUDA device; there is no CPU fallback"
    return m


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x, np.float32)).cuda()


def make_ir(rng, n, L):
    return (rng.uniform(-1, 1, (n, L)) / np.sqrt(L)).astype(np.float32)


def padded(h, L):
    out = np.zeros((h.shape[0], L), np.float32)
    out[:, :h.shape[1]] = h
    return out


def run(cf, ctx, x, B, events=None, stream=None):
    """Feeds x [channels, T*B] (device) block by block; events[t](ctx) runs before call t.  Returns the output."""
    channels, total = x.shape
    y = torch.full_like(x, float("nan"))
    for t in range(total // B):
        if events and t in events:
            events[t](ctx)
        cf.fft_convolver_process(ctx, x.data_ptr() + 4 * t * B, total, y.data_ptr() + 4 * t * B, total, stream)
    torch.cuda.synchronize()
    return y


def fresh(cf, x, B, h, L, shared):
    """Output of a context created with h zero-padded to L."""
    ctx = cf.fft_convolver_create(x.shape[0], B, dev(padded(h, L)), L, 0 if shared else L)
    try:
        return run(cf, ctx, x, B)
    finally:
        cf.fft_convolver_destroy(ctx)


def setter(cf, h, shared, fade=0):
    dh = dev(h)
    return lambda ctx: cf.fft_convolver_set_ir(ctx, dh, h.shape[1], 0 if shared else h.shape[1], fade)


def largest_period(cf, ctx, B):
    return cf.fft_convolver_segments(ctx)[-1][0] // B


@pytest.mark.parametrize("shared", [False, True])
@pytest.mark.parametrize("B", [16, 128, 1024])
def test_instant_swap_equals_a_fresh_context(cf, B, shared):
    """Swap at calls 0, 1, D - 1, D (the largest segment's first firing is call D - 1) and mid-period after it: the outputs
    before the swap are those of the old IR's context, every output from the swap on those of a context created with the new
    IR (shorter than L for per-channel IRs), bit for bit."""
    rng = np.random.default_rng(10 * B + shared)
    channels = 3
    for L in (2 * B, 3 * B + 5, BMAX + 1, 3 * BMAX - 7, 1 << 17):
        n_ir = 1 if shared else channels
        h_old = make_ir(rng, n_ir, L)
        h_new = make_ir(rng, n_ir, L if shared else max(1, 2 * L // 3))
        ctx = cf.fft_convolver_create(channels, B, dev(h_old), L, 0 if shared else L)
        D = largest_period(cf, ctx, B)
        swaps = sorted({0, 1, D - 1, D, D + D // 2, 3})
        T = max(swaps) + 2 * D + 3
        x = dev(rng.uniform(-1, 1, (channels, T * B)))
        y_old, y_new = fresh(cf, x, B, h_old, L, shared), fresh(cf, x, B, h_new, L, shared)
        try:
            for t0 in swaps:
                cf.fft_convolver_reset(ctx)
                y = run(cf, ctx, x, B, {t0: setter(cf, h_new, shared)})
                n0 = t0 * B
                assert torch.equal(y[:, :n0], y_old[:, :n0]), (L, t0)
                assert torch.equal(y[:, n0:], y_new[:, n0:]), (L, t0)
                cf.fft_convolver_set_ir(ctx, dev(h_old), L, 0 if shared else L)  # back to the old IR for the next swap point
        finally:
            cf.fft_convolver_destroy(ctx)


def rel_l2(a, b):
    return float(np.linalg.norm(np.asarray(a, np.float64) - b) / np.linalg.norm(b))


@pytest.mark.parametrize("B,L,shared", [(16, 32, True), (128, 3 * BMAX - 7, False), (1024, 1 << 17, True), (64, 5000, False)])
def test_crossfade(cf, B, L, shared):
    """fade_blocks in {1, 3, D + 2}: during the fade the output is the float64 mix (1 - g) h_old*x + g h_new*x with
    g[n] = (n - t0 B + 1) / (fade_blocks B), within 1e-5 relative L2; before it the old context's output and after it the
    new context's, bit for bit."""
    rng = np.random.default_rng(B + L)
    channels = 3
    n_ir = 1 if shared else channels
    h_old, h_new = make_ir(rng, n_ir, L), make_ir(rng, n_ir, L)
    ctx = cf.fft_convolver_create(channels, B, dev(h_old), L, 0 if shared else L)
    D = largest_period(cf, ctx, B)
    fades = (1, 3, D + 2)
    t0 = D + D // 2 + 1
    T = t0 + max(fades) + 2 * D + 3
    xh = rng.uniform(-1, 1, (channels, T * B)).astype(np.float32)
    x = dev(xh)
    y_old, y_new = fresh(cf, x, B, h_old, L, shared), fresh(cf, x, B, h_new, L, shared)
    lin_old = linear(xh, np.broadcast_to(h_old, (channels, L)))
    lin_new = linear(xh, np.broadcast_to(h_new, (channels, L)))
    try:
        for F in fades:
            cf.fft_convolver_reset(ctx)
            y = run(cf, ctx, x, B, {t0: setter(cf, h_new, shared, F)})
            n0, n1 = t0 * B, (t0 + F) * B
            assert torch.equal(y[:, :n0], y_old[:, :n0]), F
            assert torch.equal(y[:, n1:], y_new[:, n1:]), F
            g = np.clip((np.arange(n0, n1) - n0 + 1) / (F * B), 0, 1)
            want = (1 - g) * lin_old[:, n0:n1] + g * lin_new[:, n0:n1]
            err = rel_l2(y[:, n0:n1].cpu().numpy(), want)
            assert err < 1e-5, (F, err)
            cf.fft_convolver_set_ir(ctx, dev(h_old), L, 0 if shared else L)
    finally:
        cf.fft_convolver_destroy(ctx)


def test_repeated_swaps_and_reset_during_a_fade(cf):
    """A fade, an instant swap and a fade to a shorter IR: after each swap is complete the output is the fresh context's of
    that IR.  A reset during a fade ends it at the new IR: the following run is the fresh new-IR context's from call 0."""
    B, L, channels = 64, 40000, 3
    rng = np.random.default_rng(5)
    D = BMAX // B
    hs = [make_ir(rng, channels, L), make_ir(rng, channels, L), make_ir(rng, channels, L), make_ir(rng, channels, L // 3)]
    T = 700 + D + 2 + 2 * D + 5
    x = dev(rng.uniform(-1, 1, (channels, T * B)))
    ctx = cf.fft_convolver_create(channels, B, dev(hs[0]), L, L)
    try:
        y = run(cf, ctx, x, B, {100: setter(cf, hs[1], False, 3), 300: setter(cf, hs[2], False), 700: setter(cf, hs[3], False, D + 2)})
        refs = [fresh(cf, x, B, h, L, False) for h in hs]
        for ref, (a, b) in zip(refs, [(0, 100), (103, 300), (300, 700), (700 + D + 2, T)]):
            assert torch.equal(y[:, a * B:b * B], ref[:, a * B:b * B]), (a, b)
        cf.fft_convolver_reset(ctx)
        h5 = make_ir(rng, channels, L)
        run(cf, ctx, x[:, :60 * B].contiguous(), B, {50: setter(cf, h5, False, 20)})
        cf.fft_convolver_reset(ctx)
        y = run(cf, ctx, x, B)
        assert torch.equal(y, fresh(cf, x, B, h5, L, False))
        setter(cf, hs[0], False, 2)(ctx)  # the fade was cancelled: a new one is accepted
    finally:
        cf.fft_convolver_destroy(ctx)


def test_plain_calls_and_memory_are_unchanged_after_a_swap(cf):
    """Launches per plain call over a full period are the same before and after a completed swap, and a second set_ir
    allocates no device memory."""
    B, L, channels = 128, 3 * BMAX + 11, 4
    rng = np.random.default_rng(3)
    D = BMAX // B
    ctx = cf.fft_convolver_create(channels, B, dev(make_ir(rng, channels, L)), L, L)
    try:
        x = dev(rng.uniform(-1, 1, (channels, D * B)))

        def launches():
            n0 = cf.launch_count()
            run(cf, ctx, x, B)
            return cf.launch_count() - n0

        before = launches()
        h1, h2 = dev(make_ir(rng, channels, L)), dev(make_ir(rng, channels, L))
        cf.fft_convolver_set_ir(ctx, h1, L, L, 5)
        launches()  # the fade and the rest of the period
        after = launches()
        assert after == before
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info()[0]
        cf.fft_convolver_set_ir(ctx, h2, L, L, 0)
        torch.cuda.synchronize()
        assert torch.cuda.mem_get_info()[0] == free0
    finally:
        cf.fft_convolver_destroy(ctx)


def test_set_ir_is_stream_ordered(cf):
    """The new IR is written by torch on a side stream behind a long kernel; set_ir and process queued on that stream with no
    host synchronisation give the same output as the run with the IR in place before the call."""
    B, L, channels = 128, 2 * BMAX + 3, 3
    rng = np.random.default_rng(11)
    D = BMAX // B
    T = 3 * D
    h0, h1 = make_ir(rng, channels, L), make_ir(rng, channels, L)
    x = dev(rng.uniform(-1, 1, (channels, T * B)))
    t0 = D + 7
    ctx = cf.fft_convolver_create(channels, B, dev(h0), L, L)
    try:
        want = run(cf, ctx, x, B, {t0: setter(cf, h1, False, 4)})
        cf.fft_convolver_reset(ctx)
        cf.fft_convolver_set_ir(ctx, dev(h0), L, L)
        src = dev(h1)
        dst = torch.zeros_like(src)
        torch.cuda.synchronize()
        s = torch.cuda.Stream()

        def late_ir(c):
            with torch.cuda.stream(s):
                torch.cuda._sleep(20_000_000)
                dst.copy_(src)
            cf.fft_convolver_set_ir(c, dst, L, L, 4, s)

        with torch.cuda.stream(s):
            got = run(cf, ctx, x, B, {t0: late_ir}, stream=s)
        assert torch.equal(got, want)
    finally:
        cf.fft_convolver_destroy(ctx)


def test_bad_arguments_are_rejected_and_the_context_continues(cf):
    """Every bad argument, and a call during a fade, raises FFTError and leaves the context running bit-identically."""
    B, L, channels = 128, 5000, 2
    rng = np.random.default_rng(2)
    h0, h1 = make_ir(rng, channels, L), make_ir(rng, channels, L)
    d1 = dev(h1)
    x = dev(rng.uniform(-1, 1, (channels, 200 * B)))
    ctx = cf.fft_convolver_create(channels, B, dev(h0), L, L)
    shared_ctx = cf.fft_convolver_create(channels, B, dev(h0[:1]), L, 0)
    bad = [dict(ir=0), dict(ir_length=0), dict(ir_length=L + 1), dict(ir_channel_stride=L - 1), dict(ir_channel_stride=0),
           dict(fade_blocks=-1), dict(fade_blocks=(1 << 24) // B + 1), dict(ir=h1), dict(ir=d1.data_ptr() + 2)]

    def rejects(c):
        for b in bad:
            args = dict(ir=d1, ir_length=L, ir_channel_stride=L, fade_blocks=0) | b
            with pytest.raises(cf.FFTError):
                cf.fft_convolver_set_ir(c, **args)
        with pytest.raises(cf.FFTError):
            cf.fft_convolver_set_ir(shared_ctx, d1, L, L)  # shared IR: the stride must be 0
        with pytest.raises(cf.FFTError):
            cf.fft_convolver_set_ir(0, d1, L, L)

    def fade_then_reject(c):
        cf.fft_convolver_set_ir(c, d1, L, L, 6)
        with pytest.raises(cf.FFTError):
            cf.fft_convolver_set_ir(c, d1, L, L, 0)

    def during(c):
        with pytest.raises(cf.FFTError):
            cf.fft_convolver_set_ir(c, d1, L, L, 2)
        rejects(c)

    try:
        want = run(cf, ctx, x, B, {100: setter(cf, h1, False, 6)})
        cf.fft_convolver_reset(ctx)
        cf.fft_convolver_set_ir(ctx, dev(h0), L, L)
        got = run(cf, ctx, x, B, {3: rejects, 100: fade_then_reject, 103: during, 150: rejects})
        assert torch.equal(got, want)
    finally:
        cf.fft_convolver_destroy(ctx)
        cf.fft_convolver_destroy(shared_ctx)


SAN = shutil.which("compute-sanitizer", path=os.pathsep.join([os.environ.get("PATH", ""), "/usr/local/cuda/bin"]))
SWAP_CASE = """
import torch, chowdsp_fft_b200 as cf
B, L, C = 32, 2000, 2
g = torch.Generator(device="cuda").manual_seed(0)
h0, h1 = torch.rand(C, L, device="cuda", generator=g) / L, torch.rand(C, L // 2, device="cuda", generator=g) / L
x, y = torch.rand(C, 80 * B, device="cuda", generator=g), torch.empty(C, 80 * B, device="cuda")
cf.set_tuning("convolver_max_block", 256)
ctx = cf.fft_convolver_create(C, B, h0, L, L)
cf.set_tuning("convolver_max_block", -1)
for t in range(80):
    if t == 13:
        cf.fft_convolver_set_ir(ctx, h1, L // 2, L // 2, 5)
    if t == 40:
        cf.fft_convolver_set_ir(ctx, h0, L, L, 0)
    cf.fft_convolver_process(ctx, x.data_ptr() + 4 * t * B, 80 * B, y.data_ptr() + 4 * t * B, 80 * B)
torch.cuda.synchronize()
cf.fft_convolver_destroy(ctx)
print("swap case ok")
"""


@pytest.mark.parametrize("tool", ["memcheck", "racecheck"])
def test_swap_under_compute_sanitizer(tmp_path, tool):
    """One small swap-plus-fade case (re-prime, FROM_FDL, EMIT_MIX) under compute-sanitizer; any report fails the test."""
    if SAN is None:
        pytest.skip("compute-sanitizer not available")
    cmd = [SAN, "--tool", tool, "--error-exitcode", "9", "--print-limit", "20", sys.executable, "-c", SWAP_CASE]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=1500, cwd=ROOT)
    log = r.stdout[-6000:] + "\n" + r.stderr[-3000:]
    (tmp_path / f"{tool}.log").write_text(" ".join(cmd[:-1]) + "\n" + log)
    assert r.returncode == 0, log
    assert "swap case ok" in log and ("ERROR SUMMARY: 0 errors" in log or "RACECHECK SUMMARY: 0 hazards" in log), log
