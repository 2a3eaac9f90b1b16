"""Streaming STFT contexts (fft_stft_stream_*) on the GPU: analysis fed in calls of varying size is bit-identical to
fft_stft_forward on the zero-padded concatenation and runs the same kernel; synthesis is bit-identical across chunkings and to the
offline register overlap-add kernel; analysis followed by synthesis returns the delayed input; reset, no allocation, stream
ordering, launch counts, argument errors, and one case under compute-sanitizer."""
import ctypes as C
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EINVAL = -1


@pytest.fixture(scope="module")
def cf():
    import chowdsp_fft_b200 as m

    assert m.device_available(), "GPU tests need a CUDA device; there is no CPU fallback"
    return m


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x, np.float32)).cuda()


def hann(N):
    return (0.5 - 0.5 * np.cos(2 * np.pi * np.arange(N) / N)).astype(np.float32)


def chunks(frames, maxf, seed):
    """Frame counts per call: 1, 3, 1, max_frames, then random, summing to `frames`."""
    rng = np.random.default_rng(seed)
    out, f, lead = [], 0, [1, 3, 1, maxf]
    while f < frames:
        n = lead[len(out)] if len(out) < len(lead) else int(rng.integers(1, maxf + 1))
        n = min(n, frames - f)
        out.append(n)
        f += n
    return out


def analyze_all(cf, ctx, x, hop, N, split, stream=None):
    """x [C, J hop] device -> spectra [C, J, N] (NaN-initialised) through analyze calls of `split` frames."""
    channels, total = x.shape
    J = sum(split)
    spec = torch.full((channels, J, N), float("nan"), device="cuda")
    f = 0
    for n in split:
        cf.fft_stft_stream_analyze(ctx, x.data_ptr() + 4 * f * hop, total, n, spec.data_ptr() + 4 * f * N, J * N, N, stream)
        f += n
    torch.cuda.synchronize()
    return spec


def synthesize_all(cf, ctx, spec, hop, split, stream=None):
    """spectra [C, J, N] device -> signal [C, J hop] (NaN-initialised) through synthesize calls of `split` frames."""
    channels, J, N = spec.shape
    y = torch.full((channels, J * hop), float("nan"), device="cuda")
    f = 0
    for n in split:
        cf.fft_stft_stream_synthesize(ctx, spec.data_ptr() + 4 * f * N, J * N, N, n, y.data_ptr() + 4 * f * hop, J * hop, stream)
        f += n
    torch.cuda.synchronize()
    return y


def padded(x, N, hop):
    """[C, T] -> [C, N - hop + T]: the signal the streaming analysis sees."""
    return np.concatenate([np.zeros((x.shape[0], N - hop), np.float32), x], axis=1)


ANALYSIS = [(2048, 512, True, True, 3), (2048, 512, True, False, 3), (1024, 256, True, True, 2), (1024, 256, True, False, 2),
            (512, 128, True, True, 3), (512, 128, True, False, 1), (8192, 1024, True, True, 2), (8192, 1024, True, False, 1),
            (1024, 256, False, True, 5), (1024, 256, False, False, 7)]


@pytest.mark.parametrize("N,hop,windowed,ordered,channels", ANALYSIS)
def test_analysis_equals_offline_stft(cf, oracle_mod, N, hop, windowed, ordered, channels):
    """Every spectrum == fft_stft_forward on the zero-padded concatenation, bit for bit, from the same kernel; within
    parity_tol(N) of the oracle."""
    o = oracle_mod
    maxf = 6
    split = chunks(29, maxf, N + channels)
    J = sum(split)
    rng = np.random.default_rng(N + 7 * channels)
    x = rng.uniform(-1, 1, (channels, J * hop)).astype(np.float32)
    win = hann(N) if windowed else None
    s = cf.fft_new_setup(N, cf.FFT_REAL)
    ctx = cf.fft_stft_stream_create(s, channels, hop, maxf, dev(win) if windowed else None, None, 1.0, ordered)
    try:
        kernels = set()
        spec = torch.full((channels, J, N), float("nan"), device="cuda")
        dx, f = dev(x), 0
        for n in split:
            cf.fft_stft_stream_analyze(ctx, dx.data_ptr() + 4 * f * hop, J * hop, n, spec.data_ptr() + 4 * f * N, J * N, N)
            kernels.add(cf.last_kernel())
            f += n
        torch.cuda.synchronize()
        xp = padded(x, N, hop)
        ref = torch.full_like(spec, float("nan"))
        cf.fft_stft_forward(s, dev(xp), ref, channels, J, xp.shape[1], hop, J * N, N, dev(win) if windowed else None, ordered)
        torch.cuda.synchronize()
        assert kernels == {cf.last_kernel()}, (kernels, cf.last_kernel())
        got = spec.cpu().numpy()
        assert not np.isnan(got).any()
        assert np.array_equal(got, ref.cpu().numpy())
        frames = np.stack([xp[:, j * hop:j * hop + N] for j in range(J)], axis=1).reshape(-1, N)
        if windowed:
            frames = frames * win
        want = o.np_transform(frames.astype(np.float32), N, False, 8, False, ordered).reshape(channels, J, N)
        assert o.rel_l2(got, want) < o.parity_tol(N)
    finally:
        cf.fft_stft_stream_destroy(ctx)
        cf.fft_destroy_setup(s)


SYNTHESIS = [(2048, 512, True, True), (2048, 1024, False, False), (1024, 256, True, False), (1024, 128, False, True), (512, 128, True, True),
             (512, 64, True, False), (128, 32, True, True), (128, 16, False, False), (8192, 1024, True, True), (4096, 2048, True, False)]


@pytest.mark.parametrize("N,hop,windowed,ordered", SYNTHESIS)
def test_synthesis_equals_offline_overlap_add(cf, oracle_mod, N, hop, windowed, ordered):
    """The concatenated output is bit-identical across two chunkings and to fft_istft_overlap_add through ristft_kernel,
    within 1e-6 of the default-routed offline call and within tolerance of the oracle; every sample is written once."""
    o = oracle_mod
    channels, maxf = 3, 7
    J = 31
    rng = np.random.default_rng(N + hop)
    spec = o.np_transform(rng.uniform(-1, 1, (channels * J, N)).astype(np.float32), N, False, 8, False, ordered).reshape(channels, J, N)
    win = hann(N) if windowed else None
    dwin = dev(win) if windowed else None
    s = cf.fft_new_setup(N, cf.FFT_REAL)
    dspec = dev(spec)
    outs = []
    for seed in (1, 2):
        ctx = cf.fft_stft_stream_create(s, channels, hop, maxf, None, dwin, 1.0 / N, ordered)
        try:
            outs.append(synthesize_all(cf, ctx, dspec, hop, chunks(J, maxf, seed)).cpu().numpy())
            assert "ristft_carry_kernel" in cf.last_kernel(), cf.last_kernel()
        finally:
            cf.fft_stft_stream_destroy(ctx)
    assert not np.isnan(outs[0]).any()
    assert np.array_equal(outs[0], outs[1])
    samples = (J - 1) * hop + N
    ref = torch.full((channels, samples), float("nan"), device="cuda")
    cf.set_tuning("wistft", 0)
    try:
        cf.fft_istft_overlap_add(s, dspec, ref, channels, J, J * N, N, samples, hop, dwin, 1.0 / N, ordered)
        torch.cuda.synchronize()
        assert "ristft_kernel" in cf.last_kernel(), cf.last_kernel()
    finally:
        cf.set_tuning("wistft", -1)
    assert np.array_equal(outs[0], ref.cpu().numpy()[:, :J * hop])
    cf.fft_istft_overlap_add(s, dspec, ref, channels, J, J * N, N, samples, hop, dwin, 1.0 / N, ordered)
    default = ref.cpu().numpy()[:, :J * hop]
    assert o.rel_l2(outs[0], default) < 1e-6
    want = o.np_istft_overlap_add(spec, N, hop, 8, ordered, win, 1.0 / N)[:, :J * hop]
    assert o.rel_l2(outs[0], want) < o.parity_tol(N)
    cf.fft_destroy_setup(s)


@pytest.mark.parametrize("N,ordered", [(1024, True), (2048, False), (256, True)])
def test_round_trip_returns_the_delayed_input(cf, N, ordered):
    """Hann analysis + Hann synthesis at hop N/4, scale 1/N: the output over the window-overlap sum (3/2) is the input delayed
    by N - hop.  An analysis-only and a synthesis-only context give the same output as one context doing both."""
    hop, channels, maxf = N // 4, 4, 5
    split = chunks(40, maxf, N)
    J = sum(split)
    rng = np.random.default_rng(N)
    x = rng.uniform(-1, 1, (channels, J * hop)).astype(np.float32)
    dx, dwin = dev(x), dev(hann(N))
    s = cf.fft_new_setup(N, cf.FFT_REAL)
    both = cf.fft_stft_stream_create(s, channels, hop, maxf, dwin, dwin, 1.0 / N, ordered)
    ana = cf.fft_stft_stream_create(s, channels, hop, maxf, dwin, None, 1.0, ordered)
    syn = cf.fft_stft_stream_create(s, channels, hop, maxf, None, dwin, 1.0 / N, ordered)
    try:
        spec = torch.empty((channels, maxf, N), device="cuda")
        spec2 = torch.empty_like(spec)
        y = torch.full((channels, J * hop), float("nan"), device="cuda")
        y2 = torch.full_like(y, float("nan"))
        f = 0
        for n in split:  # interleaved per call, as a real-time effect runs
            cf.fft_stft_stream_analyze(both, dx.data_ptr() + 4 * f * hop, J * hop, n, spec.data_ptr(), maxf * N, N)
            cf.fft_stft_stream_synthesize(both, spec.data_ptr(), maxf * N, N, n, y.data_ptr() + 4 * f * hop, J * hop)
            cf.fft_stft_stream_analyze(ana, dx.data_ptr() + 4 * f * hop, J * hop, n, spec2.data_ptr(), maxf * N, N)
            cf.fft_stft_stream_synthesize(syn, spec2.data_ptr(), maxf * N, N, n, y2.data_ptr() + 4 * f * hop, J * hop)
            f += n
        torch.cuda.synchronize()
        got = y.cpu().numpy()
        assert np.array_equal(got, y2.cpu().numpy())
        d = N - hop
        assert np.abs(got[:, d:] / 1.5 - x[:, :J * hop - d]).max() < 1e-5
    finally:
        for c in (both, ana, syn):
            cf.fft_stft_stream_destroy(c)
        cf.fft_destroy_setup(s)


def test_reset_returns_to_silence(cf):
    """After reset, analysis and synthesis output are bit-identical to a fresh context fed the same data."""
    N, hop, channels, maxf = 1024, 256, 3, 4
    rng = np.random.default_rng(5)
    x = dev(rng.uniform(-1, 1, (channels, 24 * hop)))
    dwin = dev(hann(N))
    s = cf.fft_new_setup(N, cf.FFT_REAL)
    a = cf.fft_stft_stream_create(s, channels, hop, maxf, dwin, dwin, 1.0 / N, True)
    b = cf.fft_stft_stream_create(s, channels, hop, maxf, dwin, dwin, 1.0 / N, True)
    try:
        split = chunks(24, maxf, 3)
        spec_a = analyze_all(cf, a, x, hop, N, split)
        synthesize_all(cf, a, spec_a, hop, split)
        cf.fft_stft_stream_reset(a)
        split = chunks(24, maxf, 4)
        spec_a = analyze_all(cf, a, x, hop, N, split)
        spec_b = analyze_all(cf, b, x, hop, N, split)
        assert torch.equal(spec_a, spec_b)
        assert torch.equal(synthesize_all(cf, a, spec_a, hop, split), synthesize_all(cf, b, spec_b, hop, split))
    finally:
        cf.fft_stft_stream_destroy(a)
        cf.fft_stft_stream_destroy(b)
        cf.fft_destroy_setup(s)


def test_no_allocation_stream_order_and_launch_budget(cf):
    """200 calls leave the free device memory unchanged; analyze launches at most 2 kernels, synthesize 1, reset none; input
    written by a kernel just before on the same non-default stream is the input that is read."""
    N, hop, channels, maxf = 2048, 512, 64, 4
    s = cf.fft_new_setup(N, cf.FFT_REAL)
    dwin = dev(hann(N))
    ctx = cf.fft_stft_stream_create(s, channels, hop, maxf, dwin, dwin, 1.0 / N, True)
    ref = cf.fft_stft_stream_create(s, channels, hop, maxf, dwin, dwin, 1.0 / N, True)
    try:
        x = torch.rand((channels, maxf * hop), device="cuda")
        spec = torch.empty((channels, maxf, N), device="cuda")
        y = torch.empty((channels, maxf * hop), device="cuda")
        for _ in range(3):  # warm-up
            cf.fft_stft_stream_analyze(ctx, x, maxf * hop, maxf, spec, maxf * N, N)
            cf.fft_stft_stream_synthesize(ctx, spec, maxf * N, N, maxf, y, maxf * hop)
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info()[0]
        for i in range(100):
            n = 1 + i % maxf
            c0 = cf.launch_count()
            cf.fft_stft_stream_analyze(ctx, x, maxf * hop, n, spec, maxf * N, N)
            c1 = cf.launch_count()
            cf.fft_stft_stream_synthesize(ctx, spec, maxf * N, N, n, y, maxf * hop)
            c2 = cf.launch_count()
            assert c1 - c0 <= 2 and c2 - c1 == 1, (c1 - c0, c2 - c1)
        c0 = cf.launch_count()
        cf.fft_stft_stream_reset(ctx)
        assert cf.launch_count() == c0
        torch.cuda.synchronize()
        assert torch.cuda.mem_get_info()[0] == free0
        # stream ordering: the input is produced by a kernel on `st` right behind a long one, then read by the call on `st`
        st = torch.cuda.Stream()
        big = torch.rand((channels, 1 << 18), device="cuda")
        src = torch.rand((8, channels, maxf * hop), device="cuda")
        torch.cuda.synchronize()
        outs, want = [], []
        with torch.cuda.stream(st):
            for k in range(8):
                xin = torch.full((channels, maxf * hop), float("nan"), device="cuda")
                torch.sin(big).sum()
                xin.copy_(src[k])
                o = torch.empty((channels, maxf, N), device="cuda")
                cf.fft_stft_stream_analyze(ctx, xin, maxf * hop, maxf, o, maxf * N, N, st)
                outs.append(o)
        torch.cuda.synchronize()
        for k in range(8):
            w = torch.empty((channels, maxf, N), device="cuda")
            cf.fft_stft_stream_analyze(ref, src[k], maxf * hop, maxf, w, maxf * N, N)
            want.append(w)
        torch.cuda.synchronize()
        for k in range(8):
            assert torch.equal(outs[k], want[k]), k
    finally:
        cf.fft_stft_stream_destroy(ctx)
        cf.fft_stft_stream_destroy(ref)
        cf.fft_destroy_setup(s)


def test_argument_errors_leave_the_context_usable(cf):
    """Each bad argument returns FFT_B200_EINVAL; the context keeps working and its output is unchanged."""
    L = cf._lib.lib()
    N, hop, channels, maxf = 1024, 256, 2, 4
    s = cf.fft_new_setup(N, cf.FFT_REAL)
    ctx_out = C.c_void_p()
    for setup, h in [(s, N // 16), (s, 3 * N // 8), (s, 0)]:
        assert L.fft_stft_stream_create(setup, channels, h, maxf, None, None, 1.0, 1, None, C.byref(ctx_out)) == EINVAL
    big, cplx, mixed = cf.fft_new_setup(16384, cf.FFT_REAL), cf.fft_new_setup(1024, cf.FFT_COMPLEX), cf.fft_new_setup(1536, cf.FFT_REAL)
    for setup, n in [(big, 16384), (cplx, 1024), (mixed, 1536)]:
        assert L.fft_stft_stream_create(setup, channels, n // 4, maxf, None, None, 1.0, 1, None, C.byref(ctx_out)) == EINVAL
    for setup in (big, cplx, mixed):
        cf.fft_destroy_setup(setup)
    assert L.fft_stft_stream_create(s, channels, hop, 0, None, None, 1.0, 1, None, C.byref(ctx_out)) == EINVAL
    rng = np.random.default_rng(9)
    x = dev(rng.uniform(-1, 1, (channels, 40 * hop)))
    good = cf.fft_stft_stream_create(s, channels, hop, maxf, dev(hann(N)), dev(hann(N)), 1.0 / N, False)
    ctx = cf.fft_stft_stream_create(s, channels, hop, maxf, dev(hann(N)), dev(hann(N)), 1.0 / N, False)
    try:
        spec = torch.empty((channels, maxf, N + 8), device="cuda")
        y = torch.empty((channels, maxf * hop + 4), device="cuda")
        hx, hspec = np.zeros((channels, maxf * hop), np.float32), np.zeros((channels, maxf, N), np.float32)
        xs, ss, ys = x.data_ptr(), spec.data_ptr(), y.data_ptr()
        ws, sc, sf, yw = 40 * hop, maxf * (N + 8), N + 8, maxf * hop + 4
        bad_analyze = [(xs, ws, 0, ss, sc, sf), (xs, ws, maxf + 1, ss, sc, sf), (hx.ctypes.data, ws, 1, ss, sc, sf),
                       (xs, ws, 1, hspec.ctypes.data, sc, sf), (xs + 4, ws, 1, ss, sc, sf), (xs, ws + 1, 1, ss, sc, sf),
                       (xs, ws, 1, ss + 8, sc, sf), (xs, ws, 2, ss, sc, sf + 2), (xs, ws, 1, ss, sc + 2, sf), (0, ws, 1, ss, sc, sf)]
        bad_synth = [(ss, sc, sf, 0, ys, yw), (ss, sc, sf, maxf + 1, ys, yw), (hspec.ctypes.data, sc, sf, 1, ys, yw),
                     (ss, sc, sf, 1, hx.ctypes.data, yw), (ss + 8, sc, sf, 1, ys, yw), (ss, sc, sf + 2, 2, ys, yw),
                     (ss, sc, sf, 1, ys + 4, yw), (ss, sc, sf, 1, ys, yw + 1), (ss, sc, sf, 1, 0, yw)]
        outs = {good: [], ctx: []}
        for t in range(10):
            n = 1 + t % maxf
            for c in (good, ctx):
                if c == ctx:
                    for a in bad_analyze:
                        assert L.fft_stft_stream_analyze(ctx, *a, None) == EINVAL, a
                    for a in bad_synth:
                        assert L.fft_stft_stream_synthesize(ctx, *a, None) == EINVAL, a
                cf.fft_stft_stream_analyze(c, xs + 4 * t * maxf * hop, ws, n, spec, sc, sf)
                cf.fft_stft_stream_synthesize(c, spec, sc, sf, n, y, yw)
                torch.cuda.synchronize()
                outs[c].append((spec[:, :n, :N].clone(), y[:, :n * hop].clone()))
        for (sa, ya), (sb, yb) in zip(outs[good], outs[ctx]):
            assert torch.equal(sa, sb) and torch.equal(ya, yb)
    finally:
        cf.fft_stft_stream_destroy(good)
        cf.fft_stft_stream_destroy(ctx)
        cf.fft_destroy_setup(s)


SAN = shutil.which("compute-sanitizer", path=os.pathsep.join([os.environ.get("PATH", ""), "/usr/local/cuda/bin"]))
STREAM_CASE = """
import torch, chowdsp_fft_b200 as cf
N, hop, C, F = 512, 128, 3, 4
s = cf.fft_new_setup(N, cf.FFT_REAL)
w = 0.5 - 0.5 * torch.cos(2 * torch.pi * torch.arange(N, device="cuda") / N)
ctx = cf.fft_stft_stream_create(s, C, hop, F, w, w, 1.0 / N, False)
x, spec, y = torch.rand(C, F * hop, device="cuda"), torch.empty(C, F, N, device="cuda"), torch.empty(C, F * hop, device="cuda")
for t in range(12):
    n = 1 + t % F
    cf.fft_stft_stream_analyze(ctx, x, F * hop, n, spec, F * N, N)
    cf.fft_stft_stream_synthesize(ctx, spec, F * N, N, n, y, F * hop)
cf.fft_stft_stream_reset(ctx)
torch.cuda.synchronize()
cf.fft_stft_stream_destroy(ctx)
print("stream case ok")
"""


@pytest.mark.parametrize("tool", ["memcheck", "racecheck"])
def test_stream_under_compute_sanitizer(tmp_path, tool):
    """One small analysis + synthesis run (ring wrap, carried tails, reset) under compute-sanitizer; any report fails the test."""
    if SAN is None:
        pytest.skip("compute-sanitizer not available")
    cmd = [SAN, "--tool", tool, "--error-exitcode", "9", "--print-limit", "20", sys.executable, "-c", STREAM_CASE]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=1500, cwd=ROOT)
    log = r.stdout[-6000:] + "\n" + r.stderr[-3000:]
    (tmp_path / f"{tool}.log").write_text(" ".join(cmd[:-1]) + "\n" + log)
    assert r.returncode == 0, log
    assert "stream case ok" in log and ("ERROR SUMMARY: 0 errors" in log or "RACECHECK SUMMARY: 0 hazards" in log), log
