"""The streaming convolver (fft_convolver_*) on the GPU, through the C ABI: true linear convolution against float64 numpy for
per-channel and shared IRs across the schedule's boundaries, bit equality with a caller-managed loop of
fft_partitioned_convolve_step when the schedule is uniform, reset, the reported schedule, and argument errors."""
import numpy as np
import pytest

from tests.test_emu_convolver import schedule_rule

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
BMAX = 16384


@pytest.fixture(scope="module")
def cf():
    import chowdsp_fft_b200 as m

    assert m.device_available(), "GPU tests need a CUDA device; there is no CPU fallback"
    return m


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x, np.float32)).cuda()


def run(cf, ctx, x, B):
    """Feeds x [channels, T*B] (device) block by block; returns the output [channels, T*B]."""
    channels, total = x.shape
    y = torch.full_like(x, float("nan"))
    for t in range(total // B):
        cf.fft_convolver_process(ctx, x.data_ptr() + 4 * t * B, total, y.data_ptr() + 4 * t * B, total)
    torch.cuda.synchronize()
    return y


def linear(x, h):
    """y_c = x_c * h_c in float64, first x.shape[1] samples (FFT convolution of the float64 signals)."""
    n = x.shape[1] + h.shape[1] - 1
    size = 1 << (n - 1).bit_length()
    y = np.fft.irfft(np.fft.rfft(x.astype(np.float64), size) * np.fft.rfft(h.astype(np.float64), size), size)
    return y[:, :x.shape[1]]


def rel_l2(a, b):
    return float(np.linalg.norm(np.asarray(a, np.float64) - b) / np.linalg.norm(b))


def _lengths(B):
    return sorted({1, 3 * B + 5, 2 * B, 2 * B + 1, BMAX, BMAX + 1, 3 * BMAX - 7, 1 << 17})


@pytest.mark.parametrize("shared", [False, True])
@pytest.mark.parametrize("B", [16, 128, 1024])
def test_streaming_linear_convolution(cf, B, shared):
    """Output == np.convolve(x, h)[:T*B] (rel. L2 1e-5) for IR lengths from 1 tap to 2^17 around the schedule's boundaries
    (2B, Bmax, Bmax + 1, lengths that are not multiples of B), over enough calls for at least two firings of the largest
    block; the schedule reported by the context is the documented rule."""
    rng = np.random.default_rng(B + shared)
    channels = 3 if B == 16 else 5
    T = 2 * BMAX // B + 3
    x = rng.uniform(-1, 1, (channels, T * B)).astype(np.float32)
    dx = dev(x)
    for L in _lengths(B):
        h = (rng.uniform(-1, 1, (1 if shared else channels, L)) / np.sqrt(L)).astype(np.float32)
        dh = dev(h)
        ctx = cf.fft_convolver_create(channels, B, dh, L, 0 if shared else L)
        try:
            assert cf.fft_convolver_segments(ctx) == [(b, p) for b, p, _ in schedule_rule(B, L, BMAX)]
            y = run(cf, ctx, dx, B).cpu().numpy()
        finally:
            cf.fft_convolver_destroy(ctx)
        want = linear(x, np.broadcast_to(h, (channels, L)))
        err = rel_l2(y, want)
        assert err < 1e-5, (B, L, shared, err)


@pytest.mark.parametrize("B,L,shared", [(128, 1000, False), (16, 300, True), (1024, 9000, False)])
def test_uniform_schedule_equals_the_step_loop(cf, B, L, shared):
    """With convolver_max_block = B the context runs one uniform segment: its output is bit-identical to a caller-managed
    loop of fft_partitioned_convolve_step (windows, delay line, IR spectra from the batched unordered transform)."""
    rng = np.random.default_rng(L)
    channels, N = 4, 2 * B
    P = -(-L // B)
    T = P + 6
    x = rng.uniform(-1, 1, (channels, T * B)).astype(np.float32)
    h = (rng.uniform(-1, 1, (1 if shared else channels, L)) / np.sqrt(L)).astype(np.float32)
    cf.set_tuning("convolver_max_block", B)
    try:
        ctx = cf.fft_convolver_create(channels, B, dev(h), L, 0 if shared else L)
    finally:
        cf.set_tuning("convolver_max_block", -1)
    try:
        assert cf.fft_convolver_segments(ctx) == [(B, P)]
        y = run(cf, ctx, dev(x), B)
    finally:
        cf.fft_convolver_destroy(ctx)
    s = cf.fft_new_setup(N, cf.FFT_REAL)
    hp = np.zeros((h.shape[0], P, N), np.float32)
    padded = np.zeros((h.shape[0], P * B), np.float32)
    padded[:, :L] = h
    hp[:, :, :B] = padded.reshape(h.shape[0], P, B)
    dh = torch.empty(h.shape[0], P, N, device="cuda")
    cf.fft_transform_batched(s, dev(hp), dh, h.shape[0] * P, N, N, cf.FFT_FORWARD, False)
    xpad = dev(np.concatenate([np.zeros((channels, B), np.float32), x], axis=1))
    fdl = torch.zeros(channels, P, N, device="cuda")
    want = torch.zeros(channels, T * B, device="cuda")
    for t in range(T):
        cf.fft_partitioned_convolve_step(s, xpad.data_ptr() + 4 * t * B, xpad.shape[1], dh, 0 if shared else P * N, fdl, P * N,
                                         want.data_ptr() + 4 * t * B, want.shape[1], channels, P, t, 1.0 / N)
    torch.cuda.synchronize()
    cf.fft_destroy_setup(s)
    assert torch.equal(y, want)


def test_reset_reproduces_the_first_run(cf):
    B, L, channels = 64, 40000, 3
    rng = np.random.default_rng(7)
    dx = dev(rng.uniform(-1, 1, (channels, (2 * BMAX // B + 5) * B)))
    ctx = cf.fft_convolver_create(channels, B, dev(rng.uniform(-1, 1, (channels, L)) / 200), L, L)
    try:
        first = run(cf, ctx, dx, B)
        cf.fft_convolver_reset(ctx)
        second = run(cf, ctx, dx, B)
    finally:
        cf.fft_convolver_destroy(ctx)
    assert not torch.isnan(first).any()
    assert torch.equal(first, second)


def test_bad_arguments_are_rejected_without_a_fault(cf):
    B, L, channels = 128, 5000, 2
    ir = torch.randn(channels, L, device="cuda")
    for bad in [dict(channels=0), dict(block_size=8), dict(block_size=100), dict(block_size=32768), dict(ir_length=0),
                dict(ir_channel_stride=L - 1), dict(ir_channel_stride=-L), dict(ir=np.zeros(L, np.float32))]:
        args = dict(channels=channels, block_size=B, ir=ir, ir_length=L, ir_channel_stride=L) | bad
        with pytest.raises(cf.FFTError):
            cf.fft_convolver_create(**args)
    with pytest.raises(cf.FFTError):
        cf.set_tuning("convolver_max_block", 100)
    ctx = cf.fft_convolver_create(channels, B, ir, L, L)
    try:
        x = torch.randn(channels, 2 * B + 2, device="cuda")
        y = torch.zeros_like(x)
        for args in [(x.data_ptr() + 4, 2 * B + 2, y, 2 * B + 2),     # input not 8-byte aligned
                     (x, 2 * B + 2, y.data_ptr() + 4, 2 * B + 2),     # output not 8-byte aligned
                     (x, 2 * B + 1, y, 2 * B + 2),                     # odd stride
                     (np.zeros((channels, B), np.float32), B, y, 2 * B + 2),  # host input
                     (x, 2 * B + 2, np.zeros((channels, B), np.float32), B),  # host output
                     (0, B, y, B)]:
            with pytest.raises(cf.FFTError):
                cf.fft_convolver_process(ctx, *args)
        with pytest.raises(cf.FFTError):
            cf.fft_convolver_process(0, x, 2 * B + 2, y, 2 * B + 2)
        cf.fft_convolver_process(ctx, x, 2 * B + 2, y, 2 * B + 2)  # the context still works
        torch.cuda.synchronize()
        assert torch.isfinite(y).all()
    finally:
        cf.fft_convolver_destroy(ctx)
