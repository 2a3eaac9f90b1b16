"""Loader for the C-ABI library (chowdsp_fft_b200/lib/libchowdsp_fft_b200.so).

The library is the product; this module only binds it.  There is no Python or CPU implementation
behind it: if the shared object is missing the import fails loudly, and if no CUDA device is usable
every plan creation raises.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# CHOWDSP_FFT_B200_LIB selects another build of the same library (A/B tuning experiments, tools/ only)
LIB_PATH = os.environ.get("CHOWDSP_FFT_B200_LIB") or os.path.join(HERE, "lib", "libchowdsp_fft_b200.so")
CSRC_DIR = os.path.join(HERE, "csrc")

_fp = C.POINTER(C.c_float)
_lib = None


def build(jobs: int = 8, verbose: bool = False) -> str:
    """Compile every CUDA translation unit for sm_100a (nvcc cross-compiles without a GPU)."""
    import subprocess

    r = subprocess.run(["make", "-C", CSRC_DIR, f"-j{jobs}"], capture_output=True, text=True)
    if verbose or r.returncode != 0:
        print(r.stdout[-4000:] + r.stderr[-4000:])
    if r.returncode != 0:
        raise RuntimeError("building libchowdsp_fft_b200.so failed")
    return LIB_PATH


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C chowdsp_fft_b200/csrc`). chowdsp_fft_b200 has no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, i, ll, b, f = C.c_void_p, C.c_int, C.c_longlong, C.c_bool, C.c_float
    sig = {
        "fft_bytes_required": (C.c_size_t, [i, i, b]),
        "fft_new_setup": (vp, [i, i, b]),
        "fft_new_setup_preallocated": (vp, [i, i, vp, b]),
        "fft_destroy_setup": (None, [vp]),
        "fft_simd_width_bytes": (i, [vp]),
        "fft_transform": (None, [vp, vp, vp, vp, i]),
        "fft_transform_unordered": (None, [vp, vp, vp, vp, i]),
        "fft_convolve_unordered": (None, [vp, vp, vp, vp, f]),
        "fft_accumulate": (None, [vp, vp, vp, vp, i]),
        "aligned_malloc": (vp, [C.c_size_t]),
        "aligned_free": (None, [vp]),
        "fft_transform_batched": (i, [vp, vp, vp, i, ll, ll, i, i, vp]),
        "fft_transform_strided": (i, [vp, vp, vp, i, i, ll, ll, ll, ll, i, i, vp]),
        "fft_stft_forward": (i, [vp, vp, vp, i, i, ll, ll, ll, ll, vp, i, vp]),
        "fft_istft_overlap_add": (i, [vp, vp, vp, i, i, ll, ll, ll, ll, vp, f, i, vp]),
        "fft_juce_perform_batched": (i, [vp, vp, vp, i, ll, ll, i, vp]),
        "fft_juce_real_forward_batched": (i, [vp, vp, i, ll, i, vp]),
        "fft_juce_real_inverse_batched": (i, [vp, vp, i, ll, vp]),
        "fft_convolve_unordered_batched": (i, [vp, vp, vp, vp, i, ll, ll, ll, f, vp]),
        "fft_accumulate_batched": (i, [vp, vp, vp, vp, ll, vp]),
        "fft_partitioned_convolve_step": (i, [vp, vp, ll, vp, ll, vp, ll, vp, ll, i, i, i, f, vp]),
        "fft_convolver_create": (i, [i, i, vp, ll, ll, vp, C.POINTER(vp)]),
        "fft_convolver_process": (i, [vp, vp, ll, vp, ll, vp]),
        "fft_convolver_set_ir": (i, [vp, vp, ll, ll, i, vp]),
        "fft_convolver_reset": (i, [vp, vp]),
        "fft_convolver_segments": (i, [vp, C.POINTER(C.c_int), C.POINTER(C.c_int), i]),
        "fft_convolver_destroy": (i, [vp]),
        "fft_stft_stream_create": (i, [vp, i, ll, i, vp, vp, f, i, vp, C.POINTER(vp)]),
        "fft_stft_stream_analyze": (i, [vp, vp, ll, i, vp, ll, ll, vp]),
        "fft_stft_stream_synthesize": (i, [vp, vp, ll, ll, i, vp, ll, vp]),
        "fft_stft_stream_reset": (i, [vp, vp]),
        "fft_stft_stream_destroy": (i, [vp]),
        "fft_dist_phase": (i, [vp, i, i, i, vp, vp, i, vp]),
        "fft_dist_phase0_peer": (i, [vp, i, i, vp, C.POINTER(vp), i, vp]),
        "fft_dist_alloc": (vp, [C.c_size_t]),
        "fft_dist_free": (None, [vp]),
        "fft_dist_ipc_export": (i, [vp, vp]),
        "fft_dist_ipc_open": (vp, [vp]),
        "fft_dist_ipc_close": (None, [vp]),
        "fft_large_factors": (i, [vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
        "fft_dist_create": (i, [vp, i, i, C.POINTER(vp)]),
        "fft_dist_blob_bytes": (C.c_size_t, []),
        "fft_dist_export": (i, [vp, vp]),
        "fft_dist_connect": (i, [vp, vp]),
        "fft_dist_transform": (i, [vp, vp, vp, i, i, i, vp]),
        "fft_dist_natural_buffer": (vp, [vp]),
        "fft_dist_status": (i, [vp]),
        "fft_dist_phase_ms": (i, [vp, _fp]),
        "fft_dist_destroy": (i, [vp]),
        "fft_b200_set_tuning": (i, [C.c_char_p, i]),
        "fft_b200_last_error": (C.c_char_p, []),
        "fft_b200_last_kernel": (C.c_char_p, []),
        "fft_b200_clear_error": (None, []),
        "fft_b200_launch_count": (C.c_ulonglong, []),
        "fft_b200_device_available": (i, []),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


EXPORTED = (
    "fft_bytes_required", "fft_new_setup", "fft_new_setup_preallocated", "fft_destroy_setup",
    "fft_simd_width_bytes", "fft_transform", "fft_transform_unordered", "fft_convolve_unordered",
    "fft_accumulate", "aligned_malloc", "aligned_free", "fft_transform_batched", "fft_transform_strided", "fft_stft_forward", "fft_istft_overlap_add", "fft_juce_perform_batched", "fft_juce_real_forward_batched", "fft_juce_real_inverse_batched",
    "fft_convolve_unordered_batched", "fft_accumulate_batched", "fft_partitioned_convolve_step", "fft_convolver_create", "fft_convolver_process", "fft_convolver_set_ir", "fft_convolver_reset", "fft_convolver_segments", "fft_convolver_destroy", "fft_stft_stream_create", "fft_stft_stream_analyze", "fft_stft_stream_synthesize", "fft_stft_stream_reset", "fft_stft_stream_destroy", "fft_dist_phase", "fft_dist_phase0_peer", "fft_dist_alloc", "fft_dist_free", "fft_dist_ipc_export", "fft_dist_ipc_open", "fft_dist_ipc_close", "fft_dist_create", "fft_dist_blob_bytes", "fft_dist_export", "fft_dist_connect", "fft_dist_transform", "fft_dist_natural_buffer", "fft_dist_status", "fft_dist_phase_ms", "fft_dist_destroy", "fft_large_factors", "fft_b200_set_tuning", "fft_b200_last_error", "fft_b200_last_kernel", "fft_b200_clear_error",
    "fft_b200_launch_count", "fft_b200_device_available",
)
