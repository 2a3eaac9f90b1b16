"""chowdsp_fft_b200 -- B200-native (sm_100a) engine behind the chowdsp_fft C API.

The product is the C-ABI shared library ``chowdsp_fft_b200/lib/libchowdsp_fft_b200.so`` (headers in
``include/``); this package is the thin host-side mirror of the reference's interface used by the
tests and the benchmark.  No CPU fallback exists.
"""
from .api import (FFT_BACKWARD, FFT_COMPLEX, FFT_FORWARD, FFT_REAL, FFTError, aligned_array, aligned_free,
                  aligned_malloc, device_available, fft_accumulate, fft_accumulate_batched, fft_bytes_required,
                  fft_convolve_unordered, fft_convolve_unordered_batched, fft_convolver_create, fft_convolver_destroy,
                  fft_convolver_process, fft_convolver_reset, fft_convolver_set_ir, fft_convolver_segments, fft_destroy_setup, fft_dist_alloc, fft_dist_free, fft_dist_ipc_close,
                  fft_dist_ipc_export, fft_dist_ipc_open, fft_dist_phase, fft_dist_phase0_peer, fft_dist_create, fft_dist_blob_bytes, fft_dist_export,
                  fft_dist_connect, fft_dist_transform, fft_dist_natural_buffer, fft_dist_status, fft_dist_phase_ms, fft_dist_destroy,
                  fft_large_factors, fft_new_setup,
                  fft_new_setup_preallocated, fft_partitioned_convolve_step, fft_simd_width_bytes, fft_stft_forward, fft_istft_overlap_add,
                  fft_stft_stream_analyze, fft_stft_stream_create, fft_stft_stream_destroy, fft_stft_stream_reset, fft_stft_stream_synthesize, fft_juce_perform_batched, fft_juce_real_forward_batched,
                  fft_juce_real_inverse_batched, fft_transform, fft_transform_batched,
                  fft_transform_strided, fft_transform_unordered, last_kernel, launch_count, set_tuning)

__all__ = [n for n in dir() if not n.startswith("_")]
