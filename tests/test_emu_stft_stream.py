"""CPU checks of streaming overlap-add synthesis (ristft_body with CARRY, behind fft_stft_stream_synthesize) through the emulator in
tests/emu (its own driver, tests/emu/emu_stft_stream_driver.cpp): a channel's frames split at random points into launches of
ristft_carry_kernel, with the carried accumulators handed from launch to launch, give a signal bit-identical to one offline
ristft_kernel run over all frames, whatever its segmentation, and the carry left behind is the offline run's tail.  One case also
runs under the ThreadSanitizer build of the emulator."""
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


def build_emu() -> str:
    """tests/emu/emu_stft_stream_driver.cpp + the kernel source, compiled for the host through tests/emu/cuda_emu.h
    (CFB_EMU_DEFINES selects a variant build, e.g. ThreadSanitizer, into a library of its own)."""
    defines = os.environ.get("CFB_EMU_DEFINES", "").split()
    so = os.path.join(EMU_DIR, "libfft_emu_stft_stream.so" if not defines else "libfft_emu_stft_stream_ab.so")
    driver = os.path.join(EMU_DIR, "emu_stft_stream_driver.cpp")
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
    L.emu_ristft_stream.argtypes = [C.c_int] * 3 + [fp, fp, C.c_int, C.c_int] + [ll] * 3 + [fp, C.c_float, C.c_int, fp]
    return L


def _p(a):
    return None if a is None else a.ctypes.data_as(fp)


def _run(emu, N, hq, logW, spec, out, channels, frames, window, nseg=1, carry=None):
    """spec: [channels][>= frames][N] view, out: [channels][samples] view (both C-contiguous per row of frames / samples)."""
    rc = emu.emu_ristft_stream(int(np.log2(N)) - 1, hq, logW, _p(spec), _p(out), channels, frames, spec.strides[0] // 4, N,
                               out.strides[0] // 4, _p(window), 1.0 / N, nseg, _p(carry))
    assert rc == 0


def _splits(rng, frames):
    cuts, f = [], 0
    while f < frames:
        n = int(min(frames - f, rng.choice([1, 1, 2, 3, 5, 8])))
        cuts.append((f, n))
        f += n
    return cuts


CASES = [(128, 2, 8, True), (128, 4, 8, False), (128, 8, 8, True), (1024, 2, 8, False), (1024, 4, 4, False), (1024, 4, 8, True),
         (1024, 8, 8, True), (4096, 2, 8, True), (4096, 4, 8, False), (4096, 8, 8, False)]


@pytest.mark.parametrize("N,hq,W,ordered", CASES)
@pytest.mark.parametrize("windowed", [False, True])
def test_carried_synthesis_is_bit_equal_to_offline(emu, oracle_mod, N, hq, W, ordered, windowed):
    """ristft_carry_kernel over random splits of the frames == ristft_kernel over all of them (nseg 1 and 3) bit for bit; every
    streamed sample is written exactly once (buffers start as NaN); the final carry == the offline signal's last N - hop samples."""
    o = oracle_mod
    channels = 3 if N >= 1024 else 21  # N = 128: several items per warp (T < 32, the uniform-iteration case), ragged last CTA
    frames = 19 if N >= 4096 else 26
    hop = hq * N // 16
    logW = 0 if ordered else {8: 3, 4: 2}[W]
    rng = np.random.default_rng(N + 10 * hq + windowed)
    x = rng.uniform(-1, 1, (channels * frames, N)).astype(np.float32)
    spec = np.ascontiguousarray(o.np_transform(x, N, False, W, False, ordered).reshape(channels, frames, N))
    win = (0.5 - 0.5 * np.cos(2 * np.pi * (np.arange(N) + 0.5) / N)).astype(np.float32) if windowed else None
    samples = (frames - 1) * hop + N
    offline = []
    for nseg in (1, 3):
        out = np.full((channels, samples + 2), np.nan, np.float32)
        _run(emu, N, hq, logW, spec, out, channels, frames, win, nseg=nseg)
        offline.append(out[:, :samples])
    assert np.array_equal(offline[0], offline[1])
    want = o.np_istft_overlap_add(spec, N, hop, W, ordered, win, 1.0 / N)
    assert o.rel_l2(offline[0], want) < min(o.parity_tol(N), 4e-7)
    for trial in range(2):
        carry = np.zeros((channels, N - hop), np.float32)
        stream = np.full((channels, frames * hop + 2), np.nan, np.float32)
        for f0, n in _splits(rng, frames):
            sub = np.ascontiguousarray(spec[:, f0:f0 + n])
            part = np.full((channels, n * hop + 2), np.nan, np.float32)
            _run(emu, N, hq, logW, sub, part, channels, n, win, carry=carry)
            assert np.all(np.isnan(part[:, n * hop:]))
            stream[:, f0 * hop:(f0 + n) * hop] = part[:, :n * hop]
        assert not np.any(np.isnan(stream[:, :frames * hop]))
        assert np.array_equal(stream[:, :frames * hop], offline[0][:, :frames * hop]), trial
        assert np.array_equal(carry, offline[0][:, frames * hop:])


@pytest.mark.timeout(900)
def test_carried_synthesis_has_no_shared_memory_races(tmp_path):
    tsan = subprocess.run(["gcc", "-print-file-name=libtsan.so"], capture_output=True, text=True).stdout.strip()
    if not (os.path.isabs(tsan) and os.path.exists(tsan)) or os.environ.get("CFB_EMU_DEFINES"):
        pytest.skip("libtsan not available (or already inside a variant build)")
    log = str(tmp_path / "tsan")
    env = dict(os.environ, CFB_EMU_DEFINES="-fsanitize=thread -g", LD_PRELOAD=tsan,
               TSAN_OPTIONS=f"halt_on_error=0 report_signal_unsafe=0 history_size=2 exitcode=0 log_path={log}")
    r = subprocess.run([sys.executable, "-m", "pytest", "tests/test_emu_stft_stream.py", "-x", "-q", "-p", "no:cacheprovider", "-k",
                        "bit_equal and True-1024-4-8-True"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=850)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert "1 passed" in r.stdout, r.stdout[-2000:]
    reports = "".join(open(f).read() for f in glob.glob(log + "*"))
    assert "ThreadSanitizer: data race" not in reports, reports[:6000]
