"""CPU checks of the kernel modes behind fft_convolver_set_ir through the emulator in tests/emu (its own driver,
tests/emu/emu_convolver_swap_driver.cpp): FROM_FDL (the newest spectrum read from the delay line instead of transformed from
the window) is bit-equal to the fused PCONV_ADD and PCONV_ADD + PARTIAL steps and leaves the delay line untouched, and
PCONV_EMIT_MIX matches a numpy restatement of the crossfade and clears the accumulator.  One case also runs under the
ThreadSanitizer build of the emulator."""
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
EMU_DIR = os.path.join(ROOT, "tests", "emu")
CSRC = os.path.join(ROOT, "chowdsp_fft_b200", "csrc")
PCONV_ADD, PCONV_EMIT, PCONV_EMIT_MIX = 1, 2, 3


def build_emu() -> str:
    """tests/emu/emu_convolver_swap_driver.cpp + the kernel source, compiled for the host through tests/emu/cuda_emu.h
    (CFB_EMU_DEFINES selects a variant build, e.g. ThreadSanitizer, into a library of its own)."""
    defines = os.environ.get("CFB_EMU_DEFINES", "").split()
    so = os.path.join(EMU_DIR, "libfft_emu_convolver_swap.so" if not defines else "libfft_emu_convolver_swap_ab.so")
    driver = os.path.join(EMU_DIR, "emu_convolver_swap_driver.cpp")
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
    L.emu_pconv_swap.argtypes = [C.c_int] * 4 + [fp, ll] * 6 + [C.c_int] * 3 + [C.c_float] * 3
    return L


def _p(a):
    return None if a is None else a.ctypes.data_as(fp)


def _case(N, seed, channels=3, P=3):
    """A window, IR spectra, a delay line with older spectra, and block index t whose slot t % P is still stale."""
    rng = np.random.default_rng(seed)
    win = rng.uniform(-1, 1, (channels, N)).astype(np.float32)
    h = rng.uniform(-0.1, 0.1, (channels, P, N)).astype(np.float32)
    fdl = rng.uniform(-1, 1, (channels, P, N)).astype(np.float32)
    S = rng.uniform(-1, 1, (channels, N)).astype(np.float32)
    return rng, win, h, fdl, S, P + 1


def _run(emu, N, W, mode, from_fdl, win, h, fdl, out, acc=None, S=None, t=4, mix=(0.0, 0.0)):
    channels, P, _ = h.shape
    B = N // 2
    logM, logW = int(np.log2(N)) - 1, {4: 2, 8: 3}[W]
    rc = emu.emu_pconv_swap(logM, logW, mode, int(from_fdl), _p(win), N, _p(h), P * N, _p(fdl), P * N, _p(out), B, _p(acc), B, _p(S), N,
                            channels, P, t, 1.0 / N, *mix)
    assert rc == 0


@pytest.mark.parametrize("N,W", [(32, 4), (256, 8)])
@pytest.mark.parametrize("partial", [False, True])
def test_from_fdl_add_is_bit_equal_to_the_fused_step(emu, N, W, partial):
    """The fused PCONV_ADD (+ PARTIAL) transforms the window and writes X_t into slot t % P; FROM_FDL on that delay line, with
    a window of NaNs it must not read, adds bit-identical values and writes nothing to the delay line."""
    rng, win, h, fdl, S, t = _case(N, N + partial)
    B = N // 2
    z = rng.uniform(-1, 1, (h.shape[0], B)).astype(np.float32)
    fused_out = z.copy()
    _run(emu, N, W, PCONV_ADD, False, win, h, fdl, fused_out, S=S if partial else None, t=t)
    written = fdl.copy()  # slot t % P now holds the window's spectrum
    out = z.copy()
    _run(emu, N, W, PCONV_ADD, True, np.full_like(win, np.nan), h, fdl, out, S=S if partial else None, t=t)
    assert np.array_equal(out, fused_out)
    assert np.array_equal(fdl, written)
    assert not np.array_equal(out, z)


@pytest.mark.parametrize("N,W", [(32, 4), (256, 8)])
def test_emit_mix_matches_the_crossfade(emu, N, W):
    """PCONV_EMIT_MIX: out[n] = (1 - g) out[n] + g (y[n] + acc[n]), g = min(start + n step, 1), and acc cleared; y + acc is
    what the fused PCONV_EMIT writes for the same state."""
    rng, win, h, fdl, _, t = _case(N, 3 * N)
    channels, B = h.shape[0], N // 2
    acc = rng.uniform(-1, 1, (channels, B)).astype(np.float32)
    emit = np.zeros((channels, B), np.float32)
    acc_emit = acc.copy()
    _run(emu, N, W, PCONV_EMIT, False, win, h, fdl, emit, acc=acc_emit, t=t)
    assert not acc_emit.any()
    n = np.arange(B, dtype=np.float64)
    for start, step in [(1.0 / (3 * B), 1.0 / (3 * B)), (0.5 + 1.0 / B, 1.0 / B), (1.0 / B, 1.0 / B)]:
        old = rng.uniform(-1, 1, (channels, B)).astype(np.float32)
        out, acc_mix = old.copy(), acc.copy()
        _run(emu, N, W, PCONV_EMIT_MIX, True, np.full_like(win, np.nan), h, fdl, out, acc=acc_mix, t=t, mix=(start, step))
        g = np.minimum(start + n * step, 1.0)
        want = (1 - g) * old.astype(np.float64) + g * emit.astype(np.float64)
        assert np.linalg.norm(out - want) / np.linalg.norm(want) < 1e-6, (start, step)
        assert not acc_mix.any()
        if start + (B - 1) * step >= 1.0:
            assert np.array_equal(out[:, -1], emit[:, -1])  # g = 1: exactly the new result


@pytest.mark.timeout(900)
def test_swap_kernels_have_no_shared_memory_races(tmp_path):
    tsan = subprocess.run(["gcc", "-print-file-name=libtsan.so"], capture_output=True, text=True).stdout.strip()
    if not (os.path.isabs(tsan) and os.path.exists(tsan)) or os.environ.get("CFB_EMU_DEFINES"):
        pytest.skip("libtsan not available (or already inside a variant build)")
    log = str(tmp_path / "tsan")
    env = dict(os.environ, CFB_EMU_DEFINES="-fsanitize=thread -g", LD_PRELOAD=tsan,
               TSAN_OPTIONS=f"halt_on_error=0 report_signal_unsafe=0 history_size=2 exitcode=0 log_path={log}")
    r = subprocess.run([sys.executable, "-m", "pytest", "tests/test_emu_convolver_swap.py", "-x", "-q", "-p", "no:cacheprovider", "-k",
                        "(bit_equal and True and 256) or (crossfade and 256)"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=850)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert "2 passed" in r.stdout, r.stdout[-2000:]
    reports = "".join(open(f).read() for f in glob.glob(log + "*"))
    assert "ThreadSanitizer: data race" not in reports, reports[:6000]
