"""CPU pre-validation of the CUDA kernel SOURCE (chowdsp_fft_b200/csrc/*.cuh) through the host shim in
tests/emu: index maps, twiddle tables, layouts, batching and shared-memory bank behaviour, checked
against the oracle.  This exercises the kernel source, not the product library; the GPU parity tests
(tests/test_gpu_parity.py, -m gpu) are the ones that go through the C ABI."""
import ctypes as C
import os

import numpy as np
import pytest

fp = C.POINTER(C.c_float)


@pytest.fixture(scope="module")
def emu():
    from tests.emu.build_emu import build

    L = C.CDLL(build())
    L.emu_fft.argtypes = [C.c_int] * 4 + [fp, fp, C.c_int, C.c_int] + [C.c_longlong] * 4 + [C.c_int, C.POINTER(C.c_long)]
    L.emu_convolve.argtypes = [fp, fp, fp] + [C.c_longlong] * 3 + [C.c_int] * 4 + [C.c_float]
    L.emu_accumulate.argtypes = [fp, fp, fp, C.c_longlong]
    L.emu_pipe.argtypes = [C.c_int, C.c_int, C.c_int, fp, fp, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_long)]
    L.emu_stft_pipe.argtypes = [C.c_int] * 4 + [fp, fp, C.c_int, C.c_int] + [C.c_longlong] * 4 + [fp, C.c_int, C.c_int, C.POINTER(C.c_long)]
    L.emu_wpipe.argtypes = [C.c_int] * 5 + [fp, fp, C.c_int, C.c_int] + [C.c_longlong] * 4 + [fp, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_long)]
    L.emu_wistft.argtypes = [C.c_int, C.c_int, fp, fp, C.c_int, C.c_int] + [C.c_longlong] * 3 + [fp, C.c_float, C.c_int, C.c_int, C.c_int]
    L.emu_istft.argtypes = [C.c_int] * 4 + [fp, fp, C.c_int, C.c_int] + [C.c_longlong] * 4 + [fp, C.c_float, C.c_int]
    L.emu_ristft.argtypes = [C.c_int] * 3 + [fp, fp, C.c_int, C.c_int] + [C.c_longlong] * 3 + [fp, C.c_float, C.c_int]
    L.emu_mixed.argtypes = [C.c_int, C.c_int, C.c_int, fp, fp, C.c_int, C.c_longlong, C.c_longlong, C.c_int]
    L.emu_mixq.argtypes = [C.c_int, C.c_int, C.c_int, fp, fp, C.c_int, C.c_longlong, C.c_longlong]
    L.emu_small.argtypes = [C.c_int, C.c_int, C.c_int, fp, fp, C.c_int, C.c_int, C.POINTER(C.c_long)]
    L.emu_fft_juce.argtypes = [C.c_int, C.c_int, C.c_int, fp, fp, C.c_int, C.c_longlong, C.c_longlong]
    L.emu_stft.argtypes = [C.c_int] * 3 + [fp, fp, C.c_int, C.c_int] + [C.c_longlong] * 4 + [fp, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_long)]
    return L


def run_fft(L, x, N, is_c, W, backward, ordered, batch, inner=None, strides=None, out_floats=None, log=False):
    logM = int(np.log2(N)) - (0 if is_c else 1)
    kind = (1 if backward else 0) if is_c else (3 if backward else 2)
    nfl = 2 * N if is_c else N
    x = np.ascontiguousarray(x, np.float32)
    out = np.zeros(out_floats if out_floats is not None else batch * nfl, np.float32)
    st = (C.c_long * 4)()
    inner = batch if inner is None else inner
    ii, io, oi, oo = strides if strides is not None else (nfl, 0, nfl, 0)
    rc = L.emu_fft(logM, kind, 0 if ordered else 1, {8: 3, 4: 2}[W], x.ctypes.data_as(fp), out.ctypes.data_as(fp),
                   batch, inner, ii, io, oi, oo, int(log), st)
    assert rc == 0
    return out, list(st)


SIZES = [(16, True), (32, True), (64, True), (256, True), (512, True), (1024, True), (4096, True), (8192, True),
         (16384, True), (32, False), (64, False), (128, False), (1024, False), (2048, False), (8192, False), (32768, False)]


@pytest.mark.parametrize("N,is_c", SIZES)
@pytest.mark.parametrize("avx", [True, False])
def test_emulated_kernels_match_oracle(emu, oracle_mod, N, is_c, avx):
    o = oracle_mod
    W = o.simd_width(N, is_c, avx)
    if W == 0 or (avx and W != 8):
        pytest.skip("layout not available at this size")
    nfl = 2 * N if is_c else N
    batch = 3 if N <= 2048 else 1  # 3 exercises the ragged last CTA for small N (several transforms per CTA)
    rng = np.random.default_rng(N + W)
    x = rng.uniform(-1, 1, (batch, nfl)).astype(np.float32)
    tol = o.parity_tol(N)  # north star: rel L2 <= 1e-6 log2 N
    for ordered in (True, False):
        f, st = run_fft(emu, x, N, is_c, W, False, ordered, batch, log=True)
        ref = o.np_transform(x, N, is_c, W, False, ordered)
        assert o.rel_l2(f, ref) < min(tol, 4e-7)
        b, st2 = run_fft(emu, ref, N, is_c, W, True, ordered, batch, log=True)
        assert o.rel_l2(b, o.np_transform(ref, N, is_c, W, True, ordered)) < min(tol, 4e-7)
        for s in (st, st2):
            if s[0]:
                M = N if is_c else N // 2
                if M >= 512:
                    # shared-memory exchanges: <= 10% extra wavefronts overall (the mirrored reads of the
                    # real split step collide on one slot per 16), nothing worse than 2x on one access
                    assert s[1] <= 1.10 * s[2], s
                    assert s[3] <= 200, s
                else:
                    # several small transforms share a warp; their staging images alias in the banks
                    assert s[1] <= 2.6 * s[2] and s[3] <= 400, s


@pytest.mark.parametrize("N,is_c", [(512, True), (1024, True), (8192, True), (16384, True), (1024, False), (2048, False), (16384, False), (32768, False)])
def test_emulated_radix32_geometry(emu, oracle_mod, N, is_c):
    """The 32-points-per-thread geometry (one exchange fewer for M = 512, 1024, 8192, 16384): same results,
    conflict-free exchanges."""
    o = oracle_mod
    W = 8
    nfl = 2 * N if is_c else N
    batch = 3 if N <= 2048 else 1
    rng = np.random.default_rng(N + 32)
    x = rng.uniform(-1, 1, (batch, nfl)).astype(np.float32)
    emu.emu_set_radix(32)
    try:
        for ordered in (True, False):
            f, st = run_fft(emu, x, N, is_c, W, False, ordered, batch, log=True)
            ref = o.np_transform(x, N, is_c, W, False, ordered)
            assert o.rel_l2(f, ref) < 4e-7
            b, st2 = run_fft(emu, ref, N, is_c, W, True, ordered, batch, log=True)
            assert o.rel_l2(b, o.np_transform(ref, N, is_c, W, True, ordered)) < 4e-7
            for s in (st, st2):
                M = N if is_c else N // 2
                if M >= 1024:
                    assert s[1] <= 1.10 * s[2] and s[3] <= 200, s
    finally:
        emu.emu_set_radix(16)


@pytest.mark.parametrize("ordered", [True, False])
@pytest.mark.parametrize("N,is_c", [(8192, True), (16384, True), (16384, False), (32768, False)])
def test_emulated_pipelined_kernel(emu, oracle_mod, N, is_c, ordered):
    """The persistent TMA-pipelined kernel (2^13 / 2^14 complex points): 3 transforms on 2 resident CTAs, so one
    CTA runs two loop iterations (landing-buffer reuse, barrier phases) and the other one; ordered and 8-lane
    unordered layouts."""
    o = oracle_mod
    nfl = 2 * N if is_c else N
    logM = int(np.log2(N)) - (0 if is_c else 1)
    batch, grid = 3, 2
    rng = np.random.default_rng(N + 77)
    x = rng.uniform(-1, 1, (batch, nfl)).astype(np.float32)
    ref = o.np_transform(x, N, is_c, 8, False, ordered)
    st = (C.c_long * 4)()
    f = np.zeros_like(x)
    assert emu.emu_pipe(logM, 0 if is_c else 2, int(not ordered), x.ctypes.data_as(fp), f.ctypes.data_as(fp), batch, grid, 1, st) == 0
    assert o.rel_l2(f, ref) < 4e-7
    assert st[1] <= 1.05 * st[2] and st[3] <= 200, list(st)
    b = np.zeros_like(x)
    refc = np.ascontiguousarray(ref, np.float32)
    assert emu.emu_pipe(logM, 1 if is_c else 3, int(not ordered), refc.ctypes.data_as(fp), b.ctypes.data_as(fp), batch, grid, 1, st) == 0
    assert o.rel_l2(b, o.np_transform(ref, N, is_c, 8, True, ordered)) < 4e-7
    assert st[1] <= 1.05 * st[2] and st[3] <= 200, list(st)


def same_bits(a, b):
    return np.array_equal(np.ascontiguousarray(a, np.float32).view(np.uint32), np.ascontiguousarray(b, np.float32).view(np.uint32))


@pytest.mark.parametrize("N,is_c", [(8192, True), (16384, True), (16384, False), (32768, False)])
def test_pipelined_kernel_bit_equal_to_fft_kernel(emu, N, is_c):
    """pipe_kernel and fft_kernel<LOGM, 32> serve the same sizes, and the dispatcher picks between them by batch geometry
    (two-level batches, row strides, alignment): a batch must give the bits of a loop of single calls whichever kernel
    runs, so the two must agree bit for bit.  Every kind, ordered and 8-lane unordered, 3 rows on 2 CTAs (one CTA loops)."""
    nfl = 2 * N if is_c else N
    logM = int(np.log2(N)) - (0 if is_c else 1)
    batch = 3
    rng = np.random.default_rng(N + 13)
    x = rng.uniform(-1, 1, (batch, nfl)).astype(np.float32)
    emu.emu_set_radix(32)
    try:
        for ordered in (True, False):
            for backward in (False, True):
                kind = (1 if backward else 0) if is_c else (3 if backward else 2)
                p = np.zeros_like(x)
                assert emu.emu_pipe(logM, kind, int(not ordered), x.ctypes.data_as(fp), p.ctypes.data_as(fp), batch, 2, 0, None) == 0
                f, _ = run_fft(emu, x, N, is_c, 8, backward, ordered, batch)
                diff = int((p.reshape(-1) != f).sum())
                assert same_bits(p.reshape(-1), f), f"ordered={ordered} backward={backward}: {diff} of {f.size} floats differ"
    finally:
        emu.emu_set_radix(16)


@pytest.mark.parametrize("N,is_c", [(512, True), (1024, True), (1024, False), (2048, False)])
def test_warp_pipelined_kernel_bit_equal_to_fft_kernel(emu, N, is_c):
    """wpipe_kernel takes plain batches of its sizes (unordered R2C 2048 from 4096 rows on) where fft_kernel takes smaller
    ones: at the same points per thread the two must agree bit for bit.  Forward kinds, every layout."""
    nfl = 2 * N if is_c else N
    logM = int(np.log2(N)) - (0 if is_c else 1)
    radix = 32 if logM == 10 else 16
    batch = 5
    rng = np.random.default_rng(N + 17)
    x = rng.uniform(-1, 1, (batch, nfl)).astype(np.float32)
    emu.emu_set_radix(radix)
    try:
        for ordered, W in ((True, 8), (False, 8), (False, 4)):
            w = np.zeros_like(x)
            rc = emu.emu_wpipe(logM, radix, 0 if is_c else 2, int(not ordered), {8: 3, 4: 2}[W], x.ctypes.data_as(fp), w.ctypes.data_as(fp),
                               1, batch, 0, nfl, 0, nfl, None, 2, 2, 0, None)
            assert rc == 0
            f, _ = run_fft(emu, x, N, is_c, W, False, ordered, batch)
            assert same_bits(w.reshape(-1), f), f"ordered={ordered} W={W}: {int((w.reshape(-1) != f).sum())} floats differ"
    finally:
        emu.emu_set_radix(16)


def test_emulated_impulse_and_tone_positions(emu, oracle_mod):
    """Unit impulses and single-bin tones expose index / sign / layout errors exactly."""
    o = oracle_mod
    N, W = 256, 8
    for is_c in (True, False):
        nfl = 2 * N if is_c else N
        x = np.zeros((2, nfl), np.float32)
        x[0, 0] = 1.0
        x[1, 2 if is_c else 1] = 1.0  # impulse at n = 1
        for ordered in (True, False):
            f, _ = run_fft(emu, x, N, is_c, W, False, ordered, 2)
            assert np.allclose(f.reshape(2, nfl), o.np_transform(x, N, is_c, W, False, ordered), atol=2e-6)
        n = np.arange(N)
        k0 = 37
        tone = np.cos(2 * np.pi * k0 * n / N).astype(np.float32)
        xt = np.zeros(nfl, np.float32)
        if is_c:
            xt[0::2] = tone
        else:
            xt[:] = tone
        f, _ = run_fft(emu, xt, N, is_c, W, False, True, 1)
        spec = f[0::2] + 1j * f[1::2]
        peak = np.argsort(-np.abs(spec))[:2 if is_c else 1]
        assert set(peak.tolist()) == ({k0, N - k0} if is_c else {k0})


def test_emulated_two_level_batch_is_an_stft_gather(emu, oracle_mod):
    """outer x inner addressing = overlapping frame gather (hop < N) for the STFT path."""
    o = oracle_mod
    N, W, hop, channels, frames = 128, 8, 32, 2, 5
    ch_stride = 400
    rng = np.random.default_rng(5)
    sig = rng.uniform(-1, 1, channels * ch_stride).astype(np.float32)
    out, _ = run_fft(emu, sig, N, False, W, False, True, channels * frames, inner=frames,
                     strides=(hop, ch_stride, N, frames * N), out_floats=channels * frames * N)
    out = out.reshape(channels, frames, N)
    for c in range(channels):
        for f in range(frames):
            want = o.np_transform(sig[c * ch_stride + f * hop: c * ch_stride + f * hop + N], N, False, W, False, True)
            assert o.rel_l2(out[c, f], want) < 4e-7


@pytest.mark.parametrize("is_c,W", [(False, 8), (False, 4), (True, 8), (True, 4)])
def test_emulated_convolve_and_accumulate(emu, oracle_mod, is_c, W):
    o = oracle_mod
    N = 256
    nfl = 2 * N if is_c else N
    rng = np.random.default_rng(11)
    batch = 3
    a = rng.uniform(-1, 1, (batch, nfl)).astype(np.float32)
    b = rng.uniform(-1, 1, nfl).astype(np.float32)  # shared operand (stride 0)
    ab = rng.uniform(-1, 1, (batch, nfl)).astype(np.float32)
    want = o.np_convolve(a, b[None, :], ab, N, is_c, W, 0.5 / N)
    got = ab.copy()
    emu.emu_convolve(a.ctypes.data_as(fp), b.ctypes.data_as(fp), got.ctypes.data_as(fp), nfl, 0, nfl, nfl, batch,
                     {8: 3, 4: 2}[W], 0 if is_c else 1, 0.5 / N)
    assert o.rel_l2(got, want) < 2e-7
    s = np.empty_like(a)
    emu.emu_accumulate(a.ctypes.data_as(fp), ab.ctypes.data_as(fp), s.ctypes.data_as(fp), a.size)
    assert np.array_equal(s, a + ab)


@pytest.mark.parametrize("N,W", [(256, 8), (256, 4), (32, 4), (2048, 8)])
def test_emulated_fused_partitioned_convolution(emu, oracle_mod, ref_lib, N, W):
    """pconv_kernel (forward -> P x MAC -> inverse, overlap-save) against the oracle's block-by-block
    composition and, when present, the reference API sequence itself."""
    o = oracle_mod
    emu.emu_pconv.argtypes = [C.c_int, C.c_int, fp, C.c_longlong, fp, C.c_longlong, fp, C.c_longlong, fp, C.c_longlong,
                              C.c_int, C.c_int, C.c_int, C.c_float]
    P, channels, blocks = 3, (2 if N >= 2048 else 37), 5  # 37 channels: more than one CTA of 32 / 256 channels at the small sizes, ragged
    B = N // 2
    rng = np.random.default_rng(N + W)
    x = rng.uniform(-1, 1, (channels, blocks * B)).astype(np.float32)
    ir = (rng.uniform(-1, 1, (channels, P * B)) * 0.1).astype(np.float32)
    h = np.zeros((channels, P, N), np.float32)
    for c in range(channels):
        for p in range(P):
            seg = np.zeros(N, np.float32)
            seg[:B] = ir[c, p * B:(p + 1) * B]
            h[c, p] = o.np_transform(seg, N, False, W, False, False)
    want_y, want_fdl = o.np_partitioned_convolve(x, h, N, P, W)
    xpad = np.ascontiguousarray(np.concatenate([np.zeros((channels, B), np.float32), x], axis=1))
    fdl = np.zeros((channels, P, N), np.float32)
    y = np.zeros((channels, blocks * B), np.float32)
    logM = int(np.log2(N)) - 1
    for t in range(blocks):
        win = xpad[:, t * B:]
        out = y[:, t * B:]
        rc = emu.emu_pconv(logM, {8: 3, 4: 2}[W], win.ctypes.data_as(fp), xpad.shape[1], h.ctypes.data_as(fp), P * N,
                           fdl.ctypes.data_as(fp), P * N, out.ctypes.data_as(fp), y.shape[1], channels, P, t, 1.0 / N)
        assert rc == 0
    assert o.rel_l2(fdl, want_fdl) < o.parity_tol(N)
    assert o.rel_l2(y, want_y) < 2e-6
    for c in range(channels):  # and it IS the linear convolution
        direct = np.convolve(x[c].astype(np.float64), ir[c].astype(np.float64))[:blocks * B]
        assert o.rel_l2(y[c], direct) < 5e-6
    if ref_lib is not None and W == o.simd_width(N, False, True):
        ref_y, ref_fdl, _ = ref_lib.partitioned_convolve(x, h, N, P)
        assert o.rel_l2(y, ref_y) < 2e-6


def _emu_large(emu, n, l1, l2, l3, backward, x, batch=1, logw=0, chunk_elems=0, lanes=1, log_conflicts=0):
    emu.emu_large_c2c.argtypes = [C.c_int] * 7 + [C.c_longlong, C.c_int, fp, fp, C.c_int, C.POINTER(C.c_long)]
    out = np.zeros_like(x)
    st = (C.c_long * 5)()
    rc = emu.emu_large_c2c(n, l1, l2, l3, backward, batch, logw, chunk_elems, lanes, x.ctypes.data_as(fp), out.ctypes.data_as(fp), log_conflicts, st)
    assert rc == 0
    return out, list(st)


@pytest.mark.parametrize("tile_c,tile_r", [(8, 0), (16, 0), (8, 1), (16, 1)])
@pytest.mark.parametrize("n,l1,l2,l3", [(12, 6, 0, 6), (13, 6, 0, 7), (15, 7, 0, 8), (18, 6, 6, 6), (15, 9, 0, 6), (15, 6, 0, 9), (16, 10, 0, 6), (16, 6, 0, 10)])
def test_emulated_multi_pass_transform(emu, n, l1, l2, l3, tile_c, tile_r):
    """Tile kernels + pass planning of the large-transform path (two- and three-pass four-step), with the
    factorisation forced so that small sizes exercise it; both tile widths; 16 and 32 points per thread (tile_r: the
    512- / 1024-point passes in two Stockham stages); bank-conflict free exchanges."""
    if tile_r and max(l1, l2, l3) < 9:
        pytest.skip("no 512- / 1024-point pass in this plan")
    emu.emu_set_tile_c(tile_c)
    emu.emu_set_tile_r(tile_r)
    N = 1 << n
    rng = np.random.default_rng(n)
    x = rng.uniform(-1, 1, 2 * N).astype(np.float32)
    z = x[0::2].astype(np.float64) + 1j * x[1::2]
    for backward in ((0, 1) if n <= 13 else (0,)):
        out, st = _emu_large(emu, n, l1, l2, l3, backward, x, log_conflicts=int(n <= 16))
        ref = np.fft.ifft(z) * N if backward else np.fft.fft(z)
        got = out[0::2] + 1j * out[1::2]
        assert np.linalg.norm(got - ref) / np.linalg.norm(ref) < 4e-7
        if n <= 16:
            assert st[1] <= 1.15 * st[2] and st[3] <= 150, list(st)  # (nearly) conflict free
    emu.emu_set_tile_c(0)
    emu.emu_set_tile_r(0)


@pytest.mark.parametrize("tile_c", [8, 16])
@pytest.mark.parametrize("n,l1,l2,l3,batch,chunk_elems,lanes", [(16, 8, 0, 8, 3, 0, 1), (17, 9, 0, 8, 2, 0, 1), (18, 8, 0, 10, 1, 0, 1), (18, 9, 0, 9, 2, 1 << 18, 2),
                                                                (22, 8, 6, 8, 1, 8 << 14, 2)])
def test_emulated_tma_tile_kernel(emu, n, l1, l2, l3, batch, chunk_elems, lanes, tile_c):
    """tile_tma_kernel (persistent CTAs, tensor-map TMA loads and stores, two landing slots) == tile_fft_kernel bit for bit:
    strided passes, the contiguous-row pass with its transposed store, batches, chunked launches (sub-ranges of a pass's
    tiles through ring slots) -- the emulated tensor copies follow the same dims / strides / box / coordinates the host
    encodes into the CUtensorMap (large_plan.h: build_tile_tma)."""
    if n >= 22 and (tile_c == 16 or not os.environ.get("CFB_RUN_SLOW_EMU")):
        pytest.skip("row-restricted (chunked three-pass) launches through the emulator take two minutes: CFB_RUN_SLOW_EMU=1; "
                    "tests/test_gpu_parity.py::test_tma_tile_kernel_equals_tile_fft_kernel covers them on the GPU")
    N = 1 << n
    rng = np.random.default_rng(n)
    x = rng.uniform(-1, 1, (batch, 2 * N)).astype(np.float32)
    emu.emu_set_tile_c(tile_c)
    try:
        for backward in (0, 1):
            emu.emu_set_tile_tma(0)
            want, _ = _emu_large(emu, n, l1, l2, l3, backward, x.reshape(-1), batch, 0, chunk_elems, lanes)
            emu.emu_set_tile_tma(1)
            got, _ = _emu_large(emu, n, l1, l2, l3, backward, x.reshape(-1), batch, 0, chunk_elems, lanes)
            assert np.array_equal(got, want), (n, backward)
            if n <= 18 and not backward:
                z = x[:, 0::2].astype(np.float64) + 1j * x[:, 1::2]
                ref = np.fft.fft(z, axis=-1)
                g = got.reshape(batch, 2 * N)
                assert np.linalg.norm((g[:, 0::2] + 1j * g[:, 1::2]) - ref) / np.linalg.norm(ref) < 4e-7
    finally:
        emu.emu_set_tile_tma(0)
        emu.emu_set_tile_c(0)


@pytest.mark.parametrize("n,l1,l2,l3,batch,chunk_elems,lanes", [
    (12, 6, 0, 6, 5, 2 << 12, 2),      # two-pass plan, chunks of 2 transforms (ragged last chunk), 2 ring slots
    (13, 6, 0, 7, 3, 1 << 13, 3),      # one transform per chunk, 3 ring slots
    (18, 6, 6, 6, 1, 16 << 12, 2),     # three-pass plan: A global, (B, C) on chunks of 16 k1-rows
    (18, 6, 6, 6, 2, 24 << 12, 3),     # batch of 2, 24-row chunks (64 rows: ragged last chunk), 3 slots
    (18, 6, 6, 6, 1, 1 << 20, 2),      # one chunk covers everything: stays on the caller's stream
])
@pytest.mark.parametrize("logw", [0, 3, 2])
def test_emulated_l2_chunked_schedule(emu, oracle_mod, n, l1, l2, l3, batch, chunk_elems, lanes, logw):
    if logw == 2 and (n, batch) not in ((12, 5), (18, 1)):
        pytest.skip("the 4-lane layout is checked on one two-pass and one three-pass case")
    if logw == 3 and batch == 2:
        pytest.skip("covered by the batch-1 cases")
    """The L2-chunked schedules (large_plan.h: build_large_schedule) compute the same transforms as the classic
    whole-array passes: chunk / ring-slot addressing of every launch, forward and backward, natural order and the
    unordered layouts folded into the last pass's stores / the first pass's loads (bit-exact permutation of the
    ordered result, positions from the oracle's closed form)."""
    o = oracle_mod
    N = 1 << n
    rng = np.random.default_rng(n + batch)
    x = rng.uniform(-1, 1, (batch, 2 * N)).astype(np.float32)
    z = x[:, 0::2].astype(np.float64) + 1j * x[:, 1::2]
    W = 1 << logw
    perm = o.np_unordered_map(N, True, W) if logw else None  # perm[unordered float slot] = ordered float slot
    # forward
    classic, st0 = _emu_large(emu, n, l1, l2, l3, 0, x.reshape(-1), batch)
    got, st1 = _emu_large(emu, n, l1, l2, l3, 0, x.reshape(-1), batch, logw, chunk_elems, lanes)
    classic, got = classic.reshape(batch, 2 * N), got.reshape(batch, 2 * N)
    ref = np.fft.fft(z)
    assert np.linalg.norm((classic[:, 0::2] + 1j * classic[:, 1::2]) - ref) / np.linalg.norm(ref) < 4e-7
    want = classic[:, perm] if logw else classic
    assert np.array_equal(got, want)
    assert st1[4] >= st0[4]
    # backward (unordered INPUT)
    xin = x[:, perm] if logw else x
    classic_b, _ = _emu_large(emu, n, l1, l2, l3, 1, x.reshape(-1), batch)
    got_b, _ = _emu_large(emu, n, l1, l2, l3, 1, np.ascontiguousarray(xin).reshape(-1), batch, logw, chunk_elems, lanes)
    assert np.array_equal(got_b, classic_b)


@pytest.mark.parametrize("N,hop,frames,ordered,W", [(2048, 512, 7, True, 8), (2048, 512, 4, False, 8), (2048, 2048, 5, True, 8),
                                                    (512, 96, 19, True, 8), (512, 130, 9, False, 8), (128, 32, 18, False, 8),
                                                    (32, 8, 21, True, 4), (32, 6, 40, False, 4), (8192, 1024, 3, True, 8)])
@pytest.mark.parametrize("windowed,union", [(False, True), (True, True), (True, False)])
def test_emulated_stft_gather(emu, oracle_mod, N, hop, frames, ordered, W, windowed, union):
    """Frame-gather kernel (union of the CTA's frames staged once in shared memory, optional window) ==
    a loop of single out-of-place transforms over the overlapping frames (the ragged last group included)."""
    o = oracle_mod
    channels = 2
    samples = (frames - 1) * hop + N + 6
    rng = np.random.default_rng(N + hop)
    sig = rng.uniform(-1, 1, (channels, samples)).astype(np.float32)
    win = (0.5 - 0.5 * np.cos(2 * np.pi * (np.arange(N) + 0.5) / N)).astype(np.float32)
    out = np.zeros((channels, frames, N), np.float32)
    st = (C.c_long * 4)()
    vec4 = int(hop % 4 == 0 and samples % 4 == 0)
    rc = emu.emu_stft(int(np.log2(N)) - 1, 0 if ordered else 1, {8: 3, 4: 2}[W], sig.ctypes.data_as(fp), out.ctypes.data_as(fp),
                      channels, frames, samples, hop, frames * N, N, win.ctypes.data_as(fp) if windowed else None, vec4, int(union), 1, st)
    assert rc == 0
    fr = np.stack([[sig[c, f * hop:f * hop + N] for f in range(frames)] for c in range(channels)])
    if windowed:
        fr = fr * win
    want = o.np_transform(fr.reshape(-1, N).astype(np.float32), N, False, W, False, ordered).reshape(out.shape)
    assert o.rel_l2(out, want) < min(o.parity_tol(N), 4e-7)


@pytest.mark.parametrize("N,radix,hop,frames,ordered,W", [(2048, 32, 512, 19, True, 8), (2048, 32, 512, 9, False, 8), (2048, 16, 2048, 5, True, 8),
                                                          (512, 16, 96, 19, True, 8), (512, 16, 128, 9, False, 8), (128, 16, 32, 18, False, 8),
                                                          (32, 16, 8, 21, True, 4), (32, 16, 12, 40, False, 4), (8192, 16, 1024, 3, True, 8)])
@pytest.mark.parametrize("windowed", [False, True])
def test_emulated_persistent_stft(emu, oracle_mod, N, radix, hop, frames, ordered, W, windowed):
    """Persistent TMA-fed frame gather (stft_pipe_kernel): 3 resident CTAs loop over the (channel, frame group) items,
    ragged last groups included; == a loop of single out-of-place transforms over the overlapping frames."""
    o = oracle_mod
    channels = 3
    samples = ((frames - 1) * hop + N + 7) // 4 * 4
    rng = np.random.default_rng(N + hop + 1)
    sig = rng.uniform(-1, 1, (channels, samples)).astype(np.float32)
    win = (0.5 - 0.5 * np.cos(2 * np.pi * (np.arange(N) + 0.5) / N)).astype(np.float32)
    out = np.zeros((channels, frames, N), np.float32)
    st = (C.c_long * 4)()
    rc = emu.emu_stft_pipe(int(np.log2(N)) - 1, radix, 0 if ordered else 1, {8: 3, 4: 2}[W], sig.ctypes.data_as(fp), out.ctypes.data_as(fp),
                           channels, frames, samples, hop, frames * N, N, win.ctypes.data_as(fp) if windowed else None, 3, 1, st)
    assert rc == 0
    fr = np.stack([[sig[c, f * hop:f * hop + N] for f in range(frames)] for c in range(channels)])
    if windowed:
        fr = fr * win
    want = o.np_transform(fr.reshape(-1, N).astype(np.float32), N, False, W, False, ordered).reshape(out.shape)
    assert o.rel_l2(out, want) < min(o.parity_tol(N), 4e-7)


@pytest.mark.parametrize("N,is_c,hop,frames,ordered,W,grid,warps", [(2048, False, 512, 19, True, 8, 2, 3), (2048, False, 512, 9, False, 8, 1, 4), (2048, False, 2048, 7, False, 4, 3, 1),
                                                                    (1024, False, 100, 23, True, 8, 2, 5), (1024, False, 256, 11, False, 8, 2, 2),
                                                                    (1024, True, 2048, 11, True, 8, 2, 3), (1024, True, 2048, 5, False, 8, 1, 2), (512, True, 1024, 9, True, 8, 2, 2), (512, True, 1024, 9, False, 4, 1, 13)])
@pytest.mark.parametrize("windowed", [False, True])
def test_emulated_warp_pipelined(emu, oracle_mod, N, is_c, hop, frames, ordered, W, grid, warps, windowed):
    """Warp-pipelined kernel (wpipe_kernel): every warp of `grid` resident CTAs loops over transforms w, w + warps in the
    grid, ..., its next input arriving by a warp-private bulk copy; plain batches (complex) and overlapping, optionally
    windowed frames (real), more and fewer transforms than warps; == a loop of single out-of-place transforms.  The
    shared-memory accesses of the landing-buffer reads must be conflict free."""
    o = oracle_mod
    if windowed and is_c:
        pytest.skip("windows are for real frames")
    channels = 3
    nfl = 2 * N if is_c else N
    samples = ((frames - 1) * hop + nfl + 7) // 4 * 4
    rng = np.random.default_rng(N + hop + 5)
    sig = rng.uniform(-1, 1, (channels, samples)).astype(np.float32)
    win = (0.5 - 0.5 * np.cos(2 * np.pi * (np.arange(N) + 0.5) / N)).astype(np.float32)
    out = np.zeros((channels, frames, nfl), np.float32)
    st = (C.c_long * 4)()
    logM = int(np.log2(N)) - (0 if is_c else 1)
    rc = emu.emu_wpipe(logM, 32 if logM == 10 else 16, 0 if is_c else 2, 0 if ordered else 1, {8: 3, 4: 2}[W], sig.ctypes.data_as(fp), out.ctypes.data_as(fp),
                       channels, frames, samples, hop, frames * nfl, nfl, win.ctypes.data_as(fp) if windowed else None, grid, warps, 1, st)
    assert rc == 0
    fr = np.stack([[sig[c, f * hop:f * hop + nfl] for f in range(frames)] for c in range(channels)])
    if windowed:
        fr = fr * win
    want = o.np_transform(fr.reshape(-1, nfl).astype(np.float32), N, is_c, W, False, ordered).reshape(out.shape)
    assert o.rel_l2(out, want) < min(o.parity_tol(N), 4e-7)
    if ordered:
        assert st[1] <= 1.1 * st[2], list(st)  # modelled wavefronts vs conflict-free count


@pytest.mark.parametrize("N,hop,frames,seg_frames,grid,warps", [(2048, 512, 21, 21, 1, 2), (2048, 512, 23, 8, 2, 3), (2048, 1024, 9, 4, 1, 10), (2048, 256, 30, 11, 2, 2),
                                                                (1024, 256, 19, 19, 1, 1), (1024, 512, 9, 3, 3, 2), (1024, 128, 40, 16, 2, 5)])
@pytest.mark.parametrize("windowed", [False, True])
def test_emulated_warp_pipelined_istft(emu, oracle_mod, N, hop, frames, seg_frames, grid, warps, windowed):
    """Warp-pipelined overlap-add synthesis (wistft_kernel): accumulators in registers shifting by hop per frame, segments
    with recomputed halos, channel tails, fewer and more items than warps; every output sample written exactly once (the
    buffer starts as NaN); == oracle.np_istft_overlap_add."""
    o = oracle_mod
    channels = 3
    rng = np.random.default_rng(N + hop + 7)
    x = rng.uniform(-1, 1, (channels * frames, N)).astype(np.float32)
    spec = np.ascontiguousarray(o.np_transform(x, N, False, 8, False, True).reshape(channels, frames, N))
    win = (0.5 - 0.5 * np.cos(2 * np.pi * (np.arange(N) + 0.5) / N)).astype(np.float32)
    samples = (frames - 1) * hop + N
    out = np.full((channels, samples + 6), np.nan, np.float32)
    rc = emu.emu_wistft(int(np.log2(N)) - 1, hop // 64, spec.ctypes.data_as(fp), out.ctypes.data_as(fp), channels, frames, frames * N, N, samples + 6,
                        win.ctypes.data_as(fp) if windowed else None, 1.0 / N, seg_frames, grid, warps)
    assert rc == 0
    want = o.np_istft_overlap_add(spec, N, hop, 8, True, win if windowed else None, 1.0 / N)
    assert np.all(np.isnan(out[:, samples:]))
    assert o.rel_l2(out[:, :samples], want) < min(o.parity_tol(N), 4e-7)


@pytest.mark.parametrize("N,radix,hop,frames,ordered,W,seg_groups", [(2048, 32, 512, 21, True, 8, 1), (2048, 32, 512, 21, False, 8, 2), (2048, 16, 2048, 5, True, 8, 1),
                                                                     (512, 16, 96, 19, True, 8, 1), (512, 16, 130, 9, False, 8, 4), (128, 16, 32, 70, False, 8, 1),
                                                                     (32, 16, 8, 45, True, 4, 1), (32, 16, 7, 40, False, 4, 2), (8192, 16, 1024, 5, True, 8, 2)])
@pytest.mark.parametrize("windowed", [False, True])
def test_emulated_istft_overlap_add(emu, oracle_mod, N, radix, hop, frames, ordered, W, seg_groups, windowed):
    """Overlap-add synthesis kernel == C2R of every frame, window, sum at hop distance (oracle.np_istft_overlap_add):
    segments with recomputed halos (seg_groups CTA groups per segment), ragged last groups, odd hops, every output
    sample written exactly once (the output buffer starts as NaN)."""
    o = oracle_mod
    channels = 2
    rng = np.random.default_rng(N + hop + 3)
    x = rng.uniform(-1, 1, (channels * frames, N)).astype(np.float32)
    spec = np.ascontiguousarray(o.np_transform(x, N, False, W, False, ordered).reshape(channels, frames, N))
    win = (0.5 - 0.5 * np.cos(2 * np.pi * (np.arange(N) + 0.5) / N)).astype(np.float32)
    samples = (frames - 1) * hop + N
    pad = 4 if windowed else 3  # 4 keeps the channels 16-byte aligned: 128-bit overlap-add path when hop % 4 == 0
    out = np.full((channels, samples + pad), np.nan, np.float32)
    rc = emu.emu_istft(int(np.log2(N)) - 1, radix, 0 if ordered else 1, {8: 3, 4: 2}[W], spec.ctypes.data_as(fp), out.ctypes.data_as(fp),
                       channels, frames, frames * N, N, samples + pad, hop, win.ctypes.data_as(fp) if windowed else None, 1.0 / N, seg_groups)
    assert rc == 0
    want = o.np_istft_overlap_add(spec, N, hop, W, ordered, win if windowed else None, 1.0 / N)
    assert np.all(np.isnan(out[:, samples:]))  # nothing written past the end of a channel
    assert o.rel_l2(out[:, :samples], want) < min(o.parity_tol(N), 4e-7)


@pytest.mark.parametrize("N,hq,W,ordered,frames,nseg", [(128, 4, 8, False, 23, 2), (128, 2, 8, True, 41, 3), (256, 4, 8, True, 30, 4), (512, 8, 4, False, 9, 1), (512, 4, 8, False, 26, 3),
                                                        (1024, 4, 8, True, 19, 1), (1024, 8, 8, False, 7, 1), (1024, 2, 4, False, 37, 3), (2048, 4, 8, False, 21, 2),
                                                        (2048, 2, 8, True, 33, 2), (4096, 4, 8, True, 11, 1), (4096, 8, 8, False, 9, 2), (8192, 4, 8, True, 9, 2)])
@pytest.mark.parametrize("windowed", [False, True])
def test_emulated_register_overlap_add(emu, oracle_mod, N, hq, W, ordered, frames, nseg, windowed):
    """ristft_kernel: overlap-add synthesis with the sums in the registers of the transform's own thread group (hop = N/2, N/4, N/8;
    32 .. 256 threads per transform; ordered and unordered spectra) == oracle.np_istft_overlap_add.  Segments with recomputed halos,
    odd channel counts (transform groups that leave a CTA early), every output sample written exactly once (the buffer starts as NaN)."""
    o = oracle_mod
    channels = 3 if N >= 1024 else 21  # small transforms: several items per warp, ragged last CTA
    hop = hq * N // 16  # hq = hop / (2 T), T = N / 32
    rng = np.random.default_rng(N + hq)
    x = rng.uniform(-1, 1, (channels * frames, N)).astype(np.float32)
    spec = np.ascontiguousarray(o.np_transform(x, N, False, W, False, ordered).reshape(channels, frames, N))
    win = (0.5 - 0.5 * np.cos(2 * np.pi * (np.arange(N) + 0.5) / N)).astype(np.float32)
    samples = (frames - 1) * hop + N
    out = np.full((channels, samples + 2), np.nan, np.float32)
    rc = emu.emu_ristft(int(np.log2(N)) - 1, hq, 0 if ordered else {8: 3, 4: 2}[W], spec.ctypes.data_as(fp), out.ctypes.data_as(fp), channels, frames,
                        frames * N, N, samples + 2, win.ctypes.data_as(fp) if windowed else None, 1.0 / N, nseg)
    assert rc == 0
    want = o.np_istft_overlap_add(spec, N, hop, W, ordered, win if windowed else None, 1.0 / N)
    assert np.all(np.isnan(out[:, samples:]))
    assert not np.any(np.isnan(out[:, :samples]))
    assert o.rel_l2(out[:, :samples], want) < min(o.parity_tol(N), 4e-7)


@pytest.mark.parametrize("N", [96, 192, 384, 480, 640, 768, 9216, 1536, 2000 * 0 + 1920])
@pytest.mark.parametrize("is_c", [True, False])
def test_emulated_mixed_radix(emu, oracle_mod, N, is_c):
    """Generic mixed-radix kernel (radix 4 / 2 / 3 / 5 Stockham passes) on the reference's non-power-of-two test
    sizes (test/test.cpp:279-285) and two more: every kind, ordered and both unordered layouts, 3 transforms on 2
    CTAs (so one CTA loops)."""
    o = oracle_mod
    nfl = 2 * N if is_c else N
    M = N if is_c else N // 2
    rng = np.random.default_rng(N + 11)
    x = rng.uniform(-1, 1, (3, nfl)).astype(np.float32)
    widths = sorted({o.simd_width(N, is_c, True), o.simd_width(N, is_c, False)} - {0})
    assert widths
    for W in widths:
        for ordered in (True, False):
            ref = o.np_transform(x, N, is_c, W, False, ordered)
            f = np.zeros_like(x)
            assert emu.emu_mixed(M, 0 if is_c else 2, 0 if ordered else W, x.ctypes.data_as(fp), f.ctypes.data_as(fp), 3, nfl, nfl, 2) == 0
            assert o.rel_l2(f, ref) < 4e-7, (W, ordered)
            b = np.zeros_like(x)
            refc = np.ascontiguousarray(ref, np.float32)
            assert emu.emu_mixed(M, 1 if is_c else 3, 0 if ordered else W, refc.ctypes.data_as(fp), b.ctypes.data_as(fp), 3, nfl, nfl, 2) == 0
            assert o.rel_l2(b, o.np_transform(ref, N, is_c, W, True, ordered)) < 4e-7, (W, ordered)


@pytest.mark.parametrize("logM", [4, 5])
def test_emulated_small_kernel(emu, oracle_mod, logM):
    """fft_small_kernel: dense batches of 16- / 32-point transforms staged through padded shared-memory rows (coalesced copies
    in and out, fft_core on the row; unordered inputs copied straight into the staging images).  Every kind / layout against the
    oracle, a ragged last CTA (batch not a multiple of the CTA's transforms) and in place; the staging copies and the row accesses
    of the ordered kinds are bank-conflict free."""
    o = oracle_mod
    M = 1 << logM
    rng = np.random.default_rng(logM)
    batch = 3 * (256 // (M // 16)) // 2 + 5  # one and a half CTAs
    stats = (C.c_long * 4)()
    for is_c in (True, False):
        N = M if is_c else 2 * M
        nfl = 2 * N if is_c else N
        x = rng.uniform(-1, 1, (batch, nfl)).astype(np.float32)
        W = o.simd_width(N, is_c, False)
        assert W == 4
        for ordered in (True, False):
            ref = np.ascontiguousarray(o.np_transform(x, N, is_c, W, False, ordered), np.float32)
            f = np.full_like(x, np.nan)
            assert emu.emu_small(logM, 0 if is_c else 2, 0 if ordered else 2, x.ctypes.data_as(fp), f.ctypes.data_as(fp), batch, 1, stats) == 0
            assert o.rel_l2(f, ref) < 4e-7, (is_c, ordered)
            assert stats[1] <= (1.05 if ordered else 2.0) * stats[2], ("shared-memory wavefronts", is_c, ordered, list(stats))
            g = x.copy()  # in place
            assert emu.emu_small(logM, 0 if is_c else 2, 0 if ordered else 2, g.ctypes.data_as(fp), g.ctypes.data_as(fp), batch, 0, None) == 0
            assert np.array_equal(g, f)
            b = np.full_like(x, np.nan)  # inverse from the ordered / unordered spectrum
            assert emu.emu_small(logM, 1 if is_c else 3, 0 if ordered else 2, ref.ctypes.data_as(fp), b.ctypes.data_as(fp), batch, 0, None) == 0
            assert o.rel_l2(b / N, x) < 4e-7, (is_c, ordered, "round trip")


@pytest.mark.parametrize("N", [96, 192, 384, 480, 640, 768, 9216, 160, 288, 1920, 2560])
@pytest.mark.parametrize("is_c", [True, False])
def test_emulated_mixq(emu, oracle_mod, N, is_c):
    """Q x 2^p kernel (mixq_kernels.cuh: power-of-two stages of fft_kernel + one radix-3 / 5 / 9 / 15 register butterfly) on the
    reference's non-power-of-two test sizes (test/test.cpp:279-285) and a few more, so that every odd factor and the one-stage
    (P = 16) geometry are covered: every kind, ordered and both unordered layouts, batches that do not fill the last CTA."""
    o = oracle_mod
    nfl = 2 * N if is_c else N
    M = N if is_c else N // 2
    rng = np.random.default_rng(N + 17)
    batch = 3 if M >= 256 else 7
    x = rng.uniform(-1, 1, (batch, nfl)).astype(np.float32)
    widths = sorted({o.simd_width(N, is_c, True), o.simd_width(N, is_c, False)} - {0})
    assert widths
    for W in widths:
        for ordered in (True, False):
            ref = o.np_transform(x, N, is_c, W, False, ordered)
            f = np.zeros_like(x)
            assert emu.emu_mixq(M, 0 if is_c else 2, 0 if ordered else W, x.ctypes.data_as(fp), f.ctypes.data_as(fp), batch, nfl, nfl) == 0
            assert o.rel_l2(f, ref) < 4e-7, (W, ordered)
            b = np.zeros_like(x)
            refc = np.ascontiguousarray(ref, np.float32)
            assert emu.emu_mixq(M, 1 if is_c else 3, 0 if ordered else W, refc.ctypes.data_as(fp), b.ctypes.data_as(fp), batch, nfl, nfl) == 0
            assert o.rel_l2(b, o.np_transform(ref, N, is_c, W, True, ordered)) < 4e-7, (W, ordered)


@pytest.mark.parametrize("logM,radix", [(4, 16), (7, 16), (10, 32), (11, 16)])
def test_emulated_juce_conventions(emu, oracle_mod, logM, radix):
    """fft_kernel_juce: real forward in place with Nyquist as bin N/2, real inverse and complex inverse scaled by 1/N
    (chowdsp_fft_juce.cpp:32-86 restated in oracle.np_juce_*)."""
    o = oracle_mod
    rng = np.random.default_rng(logM)
    N, batch = 2 << logM, 3
    stride = 2 * N + 4
    buf = rng.uniform(-1, 1, (batch, stride)).astype(np.float32)
    work = buf.copy()
    assert emu.emu_fft_juce(logM, radix, 2, work.ctypes.data_as(fp), work.ctypes.data_as(fp), batch, stride, stride) == 0
    want = o.np_juce_real_forward(buf, N, True)
    assert o.rel_l2(work[:, :N + 2], want[:, :N + 2]) < 4e-7
    assert np.all(work[:, 1] == 0) and np.all(work[:, N + 1] == 0) and np.array_equal(work[:, N + 2:], buf[:, N + 2:])
    assert emu.emu_fft_juce(logM, radix, 3, work.ctypes.data_as(fp), work.ctypes.data_as(fp), batch, stride, stride) == 0
    assert o.rel_l2(work[:, :N], buf[:, :N]) < 4e-7
    Nc = 1 << logM
    x = rng.uniform(-1, 1, (batch, 2 * Nc)).astype(np.float32)
    y = np.zeros_like(x)
    assert emu.emu_fft_juce(logM, radix, 1, x.ctypes.data_as(fp), y.ctypes.data_as(fp), batch, 2 * Nc, 2 * Nc) == 0
    assert o.rel_l2(y, o.np_juce_perform(x, Nc, True)) < 4e-7


def test_ab_switches_still_compile_and_agree():
    """The A/B switches kept in the kernel source (CFB_WPIPE_ALIAS, CFB_UNORD_DIRECT, CFB_SHFL_MIRROR, CFB_UNORD_REAL_DIRECT)
    select the alternative code paths measured in profiles/; build the emulator with every switch flipped (a second .so,
    tests/emu/build_emu.py) and rerun the transform, warp-pipelined and pipelined-kernel checks against the oracle in a
    subprocess, so that the alternatives stay correct while they are kept."""
    import os
    import subprocess
    import sys

    if os.environ.get("CFB_EMU_DEFINES"):
        pytest.skip("already running inside the flipped build")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, CFB_EMU_DEFINES="-DCFB_WPIPE_ALIAS=0 -DCFB_UNORD_DIRECT=0 -DCFB_SHFL_MIRROR=0 -DCFB_UNORD_REAL_DIRECT=1")
    r = subprocess.run([sys.executable, "-m", "pytest", "tests/test_emu_kernels.py", "-x", "-q", "-p", "no:cacheprovider",
                        "-k", "match_oracle or warp_pipelined or pipelined"], cwd=root, env=env, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
