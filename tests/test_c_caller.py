"""A compiled C caller of the drop-in ABI: the reference's own test loop (/root/reference/test/test.c:9-172) restated in
tests/c_caller/ref_test_restated.c against include/chowdsp_fft.h + the product .so, with the unmodified reference build
(oracle/_ref) standing in for pffft.  CPU: it compiles and links as C11.  GPU: it runs sizes 2^5 .. 2^19, real and complex,
SSE-layout / AVX-layout handles, malloc'd and pre-allocated setups, and every case is within the reference's tolerance."""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "c_caller", "ref_test_restated.c")
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libchowdsp_fft_ref.so")


def _build(tmp_path):
    from chowdsp_fft_b200 import _lib

    _lib.lib()
    exe = str(tmp_path / "ref_test_restated")
    r = subprocess.run(["gcc", "-std=c11", "-O1", "-Wall", "-Werror", f"-I{os.path.join(ROOT, 'include')}", SRC, _lib.LIB_PATH,
                        f"-Wl,-rpath,{os.path.dirname(_lib.LIB_PATH)}", "-ldl", "-lm", "-o", exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe


def test_c_caller_compiles_and_reports_missing_device(tmp_path):
    exe = _build(tmp_path)
    import chowdsp_fft_b200 as cf

    if cf.device_available() or not os.path.exists(REF_SO):
        return
    r = subprocess.run([exe, "5", "6", REF_SO], capture_output=True, text=True, env=dict(os.environ, CHOWDSP_FFT_B200_QUIET="1"), timeout=120)
    assert r.returncode == 1 and "FAIL setup" in r.stdout  # no CPU fallback: plan creation fails loudly, the caller sees NULL


@pytest.mark.gpu
def test_reference_c_test_loop_on_the_gpu(tmp_path):
    if not os.path.exists(REF_SO):
        pytest.skip("oracle/_ref/libchowdsp_fft_ref.so not built")
    exe = _build(tmp_path)
    r = subprocess.run([exe, "5", "19", REF_SO], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert "90 cases, 0 failures" in r.stdout and "Testing complete!" in r.stdout


# an installed but non-executable binary counts as absent
SAN = shutil.which("compute-sanitizer", path=os.pathsep.join([os.environ.get("PATH", ""), "/usr/local/cuda/bin"]))


@pytest.mark.gpu
@pytest.mark.parametrize("tool", ["memcheck", "racecheck"])
def test_compute_sanitizer_clean(tmp_path, tool):
    """SURVEY.md §5 row 2 on the real hardware (the CPU emulator's TSan pass does not model the async proxy): one small
    case per kernel family under compute-sanitizer; any report fails the test.  Logs are kept under the test's tmp_path."""
    if SAN is None:
        pytest.skip("compute-sanitizer not available")
    out_dir = str(tmp_path)
    cmds = {"py": [SAN, "--tool", tool, "--error-exitcode", "9", "--print-limit", "20", "python", os.path.join(ROOT, "tools", "sanitizer_cases.py")]}
    if os.path.exists(REF_SO):
        cmds["c"] = [SAN, "--tool", tool, "--error-exitcode", "9", "--print-limit", "20", _build(tmp_path), "5", "16", REF_SO]
    for name, cmd in cmds.items():
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=1500, cwd=ROOT)
        log = r.stdout[-6000:] + "\n" + r.stderr[-3000:]
        with open(os.path.join(out_dir, f"{tool}_{name}.log"), "w") as f:
            f.write(" ".join(cmd) + "\n" + log)
        assert r.returncode == 0, log
        assert "ERROR SUMMARY: 0 errors" in log or "RACECHECK SUMMARY: 0 hazards" in log, log
