"""CPU checks of the streaming convolver's kernel source (fft_convolver_*) through the emulator in tests/emu (its own driver,
tests/emu/emu_convolver_driver.cpp): the
accumulating output modes of the fused partitioned-convolution step (PCONV_ADD, PCONV_EMIT, the precomputed partial
spectrum), the sliced tail multiply-accumulate, and the partition schedule, each against a numpy restatement.  One case
also runs under the ThreadSanitizer build of the emulator, as tests/test_emu_race.py does for the other kernels."""
import ctypes as C
import glob
import os
import subprocess
import sys

import numpy as np
import pytest

fp = C.POINTER(C.c_float)
ll = C.c_longlong
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PCONV_ADD, PCONV_EMIT = 1, 2


EMU_DIR = os.path.join(ROOT, "tests", "emu")
CSRC = os.path.join(ROOT, "chowdsp_fft_b200", "csrc")


def build_emu() -> str:
    """tests/emu/emu_convolver_driver.cpp + the kernel source, compiled for the host through tests/emu/cuda_emu.h (flags of
    tests/emu/build_emu.py; CFB_EMU_DEFINES selects a variant build, e.g. ThreadSanitizer, into a library of its own)."""
    defines = os.environ.get("CFB_EMU_DEFINES", "").split()
    so = os.path.join(EMU_DIR, "libfft_emu_convolver.so" if not defines else "libfft_emu_convolver_ab.so")
    driver = os.path.join(EMU_DIR, "emu_convolver_driver.cpp")
    srcs = [driver, os.path.join(EMU_DIR, "cuda_emu.h")] + glob.glob(os.path.join(CSRC, "*.cuh")) + glob.glob(os.path.join(CSRC, "*.h"))
    if not defines and os.path.exists(so) and all(os.path.getmtime(so) >= os.path.getmtime(f) for f in srcs):
        return so
    cmd = ["g++", "-std=c++20", "-O1", "-fPIC", "-shared", "-pthread", *defines, f"-I{EMU_DIR}", f"-I{CSRC}", driver, "-o", so]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("emu build failed:\n" + r.stderr[-4000:])
    return so


@pytest.fixture(scope="module")
def emu():
    L = C.CDLL(build_emu())
    L.emu_pconv_acc.argtypes = [C.c_int] * 3 + [fp, ll, fp, ll, fp, ll, fp, ll, fp, ll, fp, ll] + [C.c_int] * 3 + [C.c_float]
    L.emu_pconv_slice.argtypes = [fp, ll, fp, ll, fp, ll] + [C.c_int] * 7
    L.emu_conv_schedule.argtypes = [C.c_int, ll, C.c_int, C.POINTER(C.c_int), C.POINTER(ll), C.POINTER(ll), C.c_int]
    return L


def _p(a):
    return None if a is None else a.ctypes.data_as(fp)


def _spectra(o, x, N, W):
    """Unordered forward spectra of zero-padded partitions: x [channels, P * N/2] -> [channels, P, N]."""
    channels, taps = x.shape
    B = N // 2
    P = taps // B
    seg = np.zeros((channels, P, N), np.float32)
    seg[:, :, :B] = x.reshape(channels, P, B)
    return np.ascontiguousarray(o.np_transform(seg.reshape(-1, N), N, False, W, False, False).reshape(channels, P, N), np.float32)


@pytest.mark.parametrize("N,W", [(32, 4), (256, 8)])
def test_emulated_accumulating_modes(emu, oracle_mod, N, W):
    """PCONV_EMIT writes y + acc and clears acc, PCONV_ADD adds y into the accumulator, and the PARTIAL variant multiplies
    only the newest spectrum on top of S = sum_{p >= 1} X_(t-p) H_p -- each equal to the uniform step's y."""
    o = oracle_mod
    P, channels, blocks = 3, 3, 5
    B, logM, logW = N // 2, int(np.log2(N)) - 1, {8: 3, 4: 2}[W]
    rng = np.random.default_rng(N)
    x = rng.uniform(-1, 1, (channels, blocks * B)).astype(np.float32)
    h = _spectra(o, (rng.uniform(-1, 1, (channels, P * B)) * 0.1).astype(np.float32), N, W)
    want_y, _ = o.np_partitioned_convolve(x, h, N, P, W)
    xpad = np.ascontiguousarray(np.concatenate([np.zeros((channels, B), np.float32), x], axis=1))
    fdl = {m: np.zeros((channels, P, N), np.float32) for m in ("emit", "add", "partial")}
    ref_fdl = np.zeros((channels, P, N), np.float32)
    for t in range(blocks):
        win = np.ascontiguousarray(xpad[:, t * B:t * B + N])
        want = want_y[:, t * B:(t + 1) * B]
        common = (win.ctypes.data_as(fp), N, h.ctypes.data_as(fp), P * N)

        acc = rng.uniform(-1, 1, (channels, B)).astype(np.float32)
        acc0, out = acc.copy(), np.zeros((channels, B), np.float32)
        assert emu.emu_pconv_acc(logM, logW, PCONV_EMIT, *common, _p(fdl["emit"]), P * N, _p(out), B, _p(acc), B, None, 0,
                                 channels, P, t, 1.0 / N) == 0
        assert o.rel_l2(out, want + acc0) < 2e-6
        assert not acc.any()

        z = rng.uniform(-1, 1, (channels, B)).astype(np.float32)
        out = z.copy()
        assert emu.emu_pconv_acc(logM, logW, PCONV_ADD, *common, _p(fdl["add"]), P * N, _p(out), B, None, 0, None, 0,
                                 channels, P, t, 1.0 / N) == 0
        assert o.rel_l2(out, want + z) < 2e-6

        ref_fdl[:, t % P] = o.np_transform(win, N, False, W, False, False)
        S = np.zeros((channels, N), np.float32)
        for p in range(1, min(t + 1, P)):
            S = o.np_convolve(ref_fdl[:, (t - p) % P], h[:, p], S, N, False, W, 1.0)
        out = z.copy()
        assert emu.emu_pconv_acc(logM, logW, PCONV_ADD, *common, _p(fdl["partial"]), P * N, _p(out), B, None, 0, _p(S), N,
                                 channels, P, t, 1.0 / N) == 0
        assert o.rel_l2(out, want + z) < 2e-6
    for m in fdl.values():  # every mode keeps the delay line like the plain step
        assert o.rel_l2(m, ref_fdl) < o.parity_tol(N)


@pytest.mark.parametrize("N,W,D,shared", [(64, 4, 4, False), (512, 8, 8, True), (512, 8, 1, False)])
def test_emulated_sliced_tail_mac(emu, oracle_mod, N, W, D, shared):
    """D slices of pconv_slice_kernel together write every bin of S = sum_{p=1}^{P-1} X_(q-p) H_p once; the sum over all
    partitions at once in numpy is the reference, including the real DC / Nyquist lanes."""
    o = oracle_mod
    P, channels = 5, 3
    rng = np.random.default_rng(N + D)
    fdl = rng.uniform(-1, 1, (channels, P, N)).astype(np.float32)
    h = rng.uniform(-1, 1, (1 if shared else channels, P, N)).astype(np.float32)
    pairs = N // 8 // D
    for q in (0, 3, 7):
        S = np.full((channels, N), np.nan, np.float32)
        for s in range(D):
            emu.emu_pconv_slice(_p(h), 0 if shared else P * N, _p(fdl), P * N, _p(S), N, channels, P, N, int(np.log2(W)), q % P,
                                s * pairs, pairs)
        want = np.zeros((channels, N), np.float32)
        for p in range(1, P):
            want = want + o.np_convolve(fdl[:, (q - p) % P], np.broadcast_to(h[:, p], (channels, N)), np.zeros((channels, N)), N,
                                        False, W, 1.0).astype(np.float64)
        assert not np.isnan(S).any()
        assert o.rel_l2(S, want) < 1e-6


def schedule_rule(B, L, Bmax):
    """The partition schedule, restated: [(block, partitions, first tap)]."""
    if L <= 2 * B or Bmax <= B:
        return [(B, -(-L // B), 0)]
    segs, bk = [(B, 2, 0)], 2 * B
    while bk < L:
        if bk >= Bmax:
            segs.append((bk, -(-(L - bk) // bk), bk))
            break
        segs.append((bk, 1, bk))
        bk *= 2
    return segs


def test_schedule_matches_the_rule(emu):
    blk, parts, start = (C.c_int * 16)(), (ll * 16)(), (ll * 16)()
    for B in (16, 32, 128, 1024, 16384):
        for Bmax in sorted({B, 2 * B, 4096, 16384} - {32768}):
            if Bmax < B or Bmax > 16384:
                continue
            for L in sorted({1, B - 1, B, B + 1, 2 * B, 2 * B + 1, 5 * B + 3, Bmax, Bmax + 1, 2 * Bmax, 2 * Bmax + 1, 1 << 16, 1 << 18, 10 ** 6}):
                n = emu.emu_conv_schedule(B, L, Bmax, blk, parts, start, 16)
                got = [(blk[i], parts[i], start[i]) for i in range(n)]
                assert got == schedule_rule(B, L, Bmax), (B, L, Bmax)
                # the segments tile the IR: contiguous, each covering P blocks, the last reaching past L - 1
                end = 0
                for bk, p, s0 in got:
                    assert s0 == end and (s0 == 0 or s0 >= bk)  # zero latency: the delay of a segment is at least its block
                    end = s0 + p * bk
                assert end >= L and end - got[-1][0] < L


@pytest.mark.timeout(900)
def test_convolver_kernels_have_no_shared_memory_races(tmp_path):
    tsan = subprocess.run(["gcc", "-print-file-name=libtsan.so"], capture_output=True, text=True).stdout.strip()
    if not (os.path.isabs(tsan) and os.path.exists(tsan)) or os.environ.get("CFB_EMU_DEFINES"):
        pytest.skip("libtsan not available (or already inside a variant build)")
    log = str(tmp_path / "tsan")
    env = dict(os.environ, CFB_EMU_DEFINES="-fsanitize=thread -g", LD_PRELOAD=tsan,
               TSAN_OPTIONS=f"halt_on_error=0 report_signal_unsafe=0 history_size=2 exitcode=0 log_path={log}")
    r = subprocess.run([sys.executable, "-m", "pytest", "tests/test_emu_convolver.py", "-x", "-q", "-p", "no:cacheprovider", "-k",
                        "(accumulating_modes and 256) or (sliced_tail and 64)"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=850)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert "2 passed" in r.stdout, r.stdout[-2000:]
    reports = "".join(open(f).read() for f in glob.glob(log + "*"))
    assert "ThreadSanitizer: data race" not in reports, reports[:6000]
