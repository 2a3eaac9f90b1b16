"""Host-side mirror of the reference's C API (chowdsp_fft.h:64-163) over libchowdsp_fft_b200.so.

Same function names, argument order and meaning as the reference; buffers may be numpy fp32 arrays
(host memory), torch CUDA tensors (device memory) or raw integer addresses.  Errors that the C API can
only signal with NULL / a sticky message are raised here as exceptions.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from ._lib import lib

FFT_FORWARD, FFT_BACKWARD = 0, 1   # chowdsp_fft.h:64-68
FFT_REAL, FFT_COMPLEX = 0, 1       # chowdsp_fft.h:71-75


class FFTError(RuntimeError):
    pass


def _last_error() -> str:
    return lib().fft_b200_last_error().decode(errors="replace")


def _check(rc: int) -> None:
    if rc != 0:
        raise FFTError(_last_error() or f"chowdsp_fft_b200 error {rc}")


def _addr(buf) -> int:
    """Address of a numpy array, torch tensor or raw int pointer (fp32, contiguous)."""
    if buf is None:
        return 0
    if isinstance(buf, int):
        return buf
    if isinstance(buf, np.ndarray):
        if buf.dtype != np.float32 or not buf.flags["C_CONTIGUOUS"]:
            raise TypeError("numpy buffers must be C-contiguous float32")
        return buf.ctypes.data
    if hasattr(buf, "data_ptr"):  # torch.Tensor without importing torch here
        if str(buf.dtype) != "torch.float32" or not buf.is_contiguous():
            raise TypeError("torch buffers must be contiguous float32")
        return buf.data_ptr()
    raise TypeError(f"unsupported buffer type {type(buf)!r}")


def _stream(stream) -> int:
    if stream is None:
        return 0
    if isinstance(stream, int):
        return stream
    return int(stream.cuda_stream)  # torch.cuda.Stream


def device_available() -> bool:
    return bool(lib().fft_b200_device_available())


def last_kernel() -> str:
    """Template instance of the transform kernel this thread launched last (diagnostic)."""
    return lib().fft_b200_last_kernel().decode(errors="replace")


def launch_count() -> int:
    return int(lib().fft_b200_launch_count())


def fft_bytes_required(N: int, transform: int, use_avx_if_available: bool = True) -> int:
    return int(lib().fft_bytes_required(N, transform, use_avx_if_available))


def fft_new_setup(N: int, transform: int, use_avx_if_available: bool = True) -> int:
    s = lib().fft_new_setup(N, transform, use_avx_if_available)
    if not s:
        raise FFTError(_last_error() or f"fft_new_setup({N}) failed")
    return s


def fft_new_setup_preallocated(N: int, transform: int, data, use_avx_if_available: bool = True) -> int:
    s = lib().fft_new_setup_preallocated(N, transform, _addr(data), use_avx_if_available)
    if not s:
        raise FFTError(_last_error() or f"fft_new_setup_preallocated({N}) failed")
    return s


def fft_destroy_setup(setup: int) -> None:
    lib().fft_destroy_setup(setup)


def fft_simd_width_bytes(setup: int) -> int:
    return int(lib().fft_simd_width_bytes(setup))


def _void_call(fn, *args) -> None:
    """The reference-shaped functions return void; surface the sticky error text as an exception."""
    lib().fft_b200_clear_error()
    fn(*args)
    err = _last_error()
    if err:
        raise FFTError(err)


def fft_transform(setup: int, input, output, work, direction: int) -> None:
    _void_call(lib().fft_transform, setup, _addr(input), _addr(output), _addr(work), direction)


def fft_transform_unordered(setup: int, input, output, work, direction: int) -> None:
    _void_call(lib().fft_transform_unordered, setup, _addr(input), _addr(output), _addr(work), direction)


def fft_convolve_unordered(setup: int, dft_a, dft_b, dft_ab, scaling: float) -> None:
    _void_call(lib().fft_convolve_unordered, setup, _addr(dft_a), _addr(dft_b), _addr(dft_ab), scaling)


def fft_accumulate(setup: int, a, b, ab, N: int) -> None:
    _void_call(lib().fft_accumulate, setup, _addr(a), _addr(b), _addr(ab), N)


def aligned_malloc(nb_bytes: int) -> int:
    p = lib().aligned_malloc(nb_bytes)
    if not p:
        raise MemoryError(f"aligned_malloc({nb_bytes})")
    return p


def aligned_free(p: int) -> None:
    lib().aligned_free(p)


def aligned_array(nfloats: int) -> np.ndarray:
    """fp32 numpy view of an aligned_malloc block (pinned + device-mapped when a GPU is present).
    Free with aligned_free(arr.ctypes.data) once no view is alive."""
    p = aligned_malloc(max(1, nfloats) * 4)
    return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_float)), shape=(nfloats,))


# ---- batched / stream-ordered extensions (chowdsp_fft_b200.h) --------------------------------------
def fft_transform_batched(setup: int, input, output, batch: int, in_stride: int, out_stride: int,
                          direction: int, ordered: bool = True, stream=None) -> None:
    _check(lib().fft_transform_batched(setup, _addr(input), _addr(output), batch, in_stride, out_stride,
                                       direction, int(ordered), _stream(stream)))


def fft_transform_strided(setup: int, input, output, outer: int, inner: int, in_outer: int, in_inner: int,
                          out_outer: int, out_inner: int, direction: int, ordered: bool = True, stream=None) -> None:
    _check(lib().fft_transform_strided(setup, _addr(input), _addr(output), outer, inner, in_outer, in_inner,
                                       out_outer, out_inner, direction, int(ordered), _stream(stream)))


def fft_stft_forward(setup: int, signal, spectra, channels: int, frames: int, channel_stride: int, hop: int,
                     out_channel_stride: int, out_frame_stride: int, window=None, ordered: bool = True, stream=None) -> None:
    """Short-time Fourier analysis (frame gather + optional window + R2C in one kernel, see chowdsp_fft_b200.h)."""
    _check(lib().fft_stft_forward(setup, _addr(signal), _addr(spectra), channels, frames, channel_stride, hop,
                                  out_channel_stride, out_frame_stride, _addr(window) if window is not None else None,
                                  int(ordered), _stream(stream)))


def fft_istft_overlap_add(setup: int, spectra, signal, channels: int, frames: int, spec_channel_stride: int, spec_frame_stride: int,
                          channel_stride: int, hop: int, window=None, scale: float = 1.0, ordered: bool = True, stream=None) -> None:
    """Overlap-add synthesis (C2R + optional window + sum at hop distance in one kernel, see chowdsp_fft_b200.h)."""
    _check(lib().fft_istft_overlap_add(setup, _addr(spectra), _addr(signal), channels, frames, spec_channel_stride, spec_frame_stride,
                                       channel_stride, hop, _addr(window) if window is not None else None, scale, int(ordered),
                                       _stream(stream)))


def fft_juce_perform_batched(setup: int, input, output, batch: int, in_stride: int, out_stride: int, inverse: bool, stream=None) -> None:
    """juce::dsp::FFT::perform semantics (chowdsp_fft_juce.cpp:32-46), batched: inverse scaled by 1/N."""
    _check(lib().fft_juce_perform_batched(setup, _addr(input), _addr(output), batch, in_stride, out_stride, int(inverse), _stream(stream)))


def fft_juce_real_forward_batched(setup: int, inout, batch: int, stride: int, ignore_negative_freqs: bool, stream=None) -> None:
    """performRealOnlyForwardTransform semantics (chowdsp_fft_juce.cpp:48-66), batched, in place."""
    _check(lib().fft_juce_real_forward_batched(setup, _addr(inout), batch, stride, int(ignore_negative_freqs), _stream(stream)))


def fft_juce_real_inverse_batched(setup: int, inout, batch: int, stride: int, stream=None) -> None:
    """performRealOnlyInverseTransform semantics (chowdsp_fft_juce.cpp:68-84), batched, in place."""
    _check(lib().fft_juce_real_inverse_batched(setup, _addr(inout), batch, stride, _stream(stream)))


def fft_convolve_unordered_batched(setup: int, dft_a, dft_b, dft_ab, batch: int, a_stride: int, b_stride: int,
                                   ab_stride: int, scaling: float, stream=None) -> None:
    _check(lib().fft_convolve_unordered_batched(setup, _addr(dft_a), _addr(dft_b), _addr(dft_ab), batch,
                                                a_stride, b_stride, ab_stride, scaling, _stream(stream)))


def fft_accumulate_batched(setup: int, a, b, ab, n: int, stream=None) -> None:
    _check(lib().fft_accumulate_batched(setup, _addr(a), _addr(b), _addr(ab), n, _stream(stream)))


def fft_partitioned_convolve_step(setup: int, windows, window_stride: int, ir, ir_channel_stride: int, fdl,
                                  fdl_channel_stride: int, output, output_stride: int, channels: int,
                                  partitions: int, block_index: int, scaling: float, stream=None) -> None:
    """One fused block step of partitioned overlap-save convolution (see chowdsp_fft_b200.h)."""
    _check(lib().fft_partitioned_convolve_step(setup, _addr(windows), window_stride, _addr(ir), ir_channel_stride,
                                               _addr(fdl), fdl_channel_stride, _addr(output), output_stride,
                                               channels, partitions, block_index, scaling, _stream(stream)))


# ---- streaming convolver with non-uniform partitions (chowdsp_fft_b200.h: fft_convolver_create ... fft_convolver_destroy) ----
def fft_convolver_create(channels: int, block_size: int, ir, ir_length: int, ir_channel_stride: int, stream=None) -> int:
    """Context that convolves `channels` signals with their IRs (ir + c*ir_channel_stride, 0 = one shared IR), block_size
    samples per channel per fft_convolver_process call, with no added latency."""
    ctx = C.c_void_p()
    _check(lib().fft_convolver_create(channels, block_size, _addr(ir), ir_length, ir_channel_stride, _stream(stream), C.byref(ctx)))
    return ctx.value


def fft_convolver_process(ctx: int, input, input_stride: int, output, output_stride: int, stream=None) -> None:
    _check(lib().fft_convolver_process(ctx, _addr(input), input_stride, _addr(output), output_stride, _stream(stream)))


def fft_convolver_set_ir(ctx: int, ir, ir_length: int, ir_channel_stride: int, fade_blocks: int = 0, stream=None) -> None:
    """Replace the context's IR while it runs: instantly (fade_blocks = 0) or with a linear crossfade over fade_blocks calls,
    keeping the reverb tail of the input already played (see chowdsp_fft_b200.h)."""
    _check(lib().fft_convolver_set_ir(ctx, _addr(ir), ir_length, ir_channel_stride, fade_blocks, _stream(stream)))


def fft_convolver_reset(ctx: int, stream=None) -> None:
    _check(lib().fft_convolver_reset(ctx, _stream(stream)))


def fft_convolver_segments(ctx: int) -> list[tuple[int, int]]:
    """The context's schedule: [(block size, partitions)] per segment."""
    n = lib().fft_convolver_segments(ctx, None, None, 0)
    _check(min(n, 0))
    blocks, parts = (C.c_int * n)(), (C.c_int * n)()
    lib().fft_convolver_segments(ctx, blocks, parts, n)
    return list(zip(blocks, parts))


def fft_convolver_destroy(ctx: int) -> None:
    _check(lib().fft_convolver_destroy(ctx))


# ---- streaming STFT (chowdsp_fft_b200.h: fft_stft_stream_create ... fft_stft_stream_destroy) ----
def fft_stft_stream_create(setup: int, channels: int, hop: int, max_frames: int, analysis_window=None, synthesis_window=None,
                           scale: float = 1.0, ordered: bool = True, stream=None) -> int:
    """Context for block-by-block STFT analysis and overlap-add synthesis of `channels` signals: hop = N/2, N/4 or N/8 of the
    REAL plan `setup` (N = 128 .. 8192), up to max_frames frames per call; the windows (None = rectangular) are copied."""
    ctx = C.c_void_p()
    _check(lib().fft_stft_stream_create(setup, channels, hop, max_frames, _addr(analysis_window), _addr(synthesis_window), scale,
                                        int(ordered), _stream(stream), C.byref(ctx)))
    return ctx.value


def fft_stft_stream_analyze(ctx: int, input, input_stride: int, frames: int, spectra, spec_channel_stride: int,
                            spec_frame_stride: int, stream=None) -> None:
    """frames * hop new samples per channel in, `frames` spectra per channel out."""
    _check(lib().fft_stft_stream_analyze(ctx, _addr(input), input_stride, frames, _addr(spectra), spec_channel_stride,
                                         spec_frame_stride, _stream(stream)))


def fft_stft_stream_synthesize(ctx: int, spectra, spec_channel_stride: int, spec_frame_stride: int, frames: int, output,
                               output_stride: int, stream=None) -> None:
    """`frames` spectra per channel in, frames * hop finished overlap-add samples per channel out."""
    _check(lib().fft_stft_stream_synthesize(ctx, _addr(spectra), spec_channel_stride, spec_frame_stride, frames, _addr(output),
                                            output_stride, _stream(stream)))


def fft_stft_stream_reset(ctx: int, stream=None) -> None:
    _check(lib().fft_stft_stream_reset(ctx, _stream(stream)))


def fft_stft_stream_destroy(ctx: int) -> None:
    _check(lib().fft_stft_stream_destroy(ctx))


def set_tuning(key: str, value: int) -> None:
    """Benchmark/sweep hook (fft_b200_set_tuning)."""
    _check(lib().fft_b200_set_tuning(key.encode(), int(value)))


def fft_large_factors(setup: int) -> tuple[int, int, int]:
    """(l1, l2, l3): log2 of the pass lengths of a multi-pass plan."""
    a, b, c = C.c_int(), C.c_int(), C.c_int()
    _check(lib().fft_large_factors(setup, C.byref(a), C.byref(b), C.byref(c)))
    return a.value, b.value, c.value


def fft_dist_phase(setup: int, phase: int, rank: int, world: int, input, output, direction: int = FFT_FORWARD, stream=None) -> None:
    """One local phase of the distributed four-step transform (see chowdsp_fft_b200.h)."""
    _check(lib().fft_dist_phase(setup, phase, rank, world, _addr(input), _addr(output), direction, _stream(stream)))


def fft_dist_phase0_peer(setup: int, rank: int, world: int, input, peer_recv: list[int], direction: int = FFT_FORWARD, stream=None) -> None:
    """Phase 0 fused with the exchange: row blocks are stored straight into the owners' buffers (peer memory)."""
    arr = (C.c_void_p * world)(*peer_recv)
    _check(lib().fft_dist_phase0_peer(setup, rank, world, _addr(input), arr, direction, _stream(stream)))


def fft_dist_alloc(nbytes: int) -> int:
    p = lib().fft_dist_alloc(nbytes)
    if not p:
        raise FFTError(_last_error() or "fft_dist_alloc failed")
    return p


def fft_dist_free(p: int) -> None:
    lib().fft_dist_free(p)


def fft_dist_ipc_export(p: int) -> bytes:
    buf = C.create_string_buffer(64)
    _check(lib().fft_dist_ipc_export(p, buf))
    return buf.raw


def fft_dist_ipc_open(handle: bytes) -> int:
    p = lib().fft_dist_ipc_open(C.create_string_buffer(handle, 64))
    if not p:
        raise FFTError(_last_error() or "fft_dist_ipc_open failed")
    return p


def fft_dist_ipc_close(p: int) -> None:
    lib().fft_dist_ipc_close(p)


# ---- the distributed transform as one call per rank (chowdsp_fft_b200.h: fft_dist_create ... fft_dist_destroy) ----
def fft_dist_create(setup: int, rank: int, world: int) -> int:
    ctx = C.c_void_p()
    _check(lib().fft_dist_create(setup, rank, world, C.byref(ctx)))
    return ctx.value


def fft_dist_blob_bytes() -> int:
    return int(lib().fft_dist_blob_bytes())


def fft_dist_export(ctx: int) -> bytes:
    buf = C.create_string_buffer(fft_dist_blob_bytes())
    _check(lib().fft_dist_export(ctx, buf))
    return buf.raw


def fft_dist_connect(ctx: int, blobs: bytes | None) -> None:
    _check(lib().fft_dist_connect(ctx, C.create_string_buffer(blobs, len(blobs)) if blobs else None))


def fft_dist_transform(ctx: int, input, output, direction: int = FFT_FORWARD, natural_order: bool = False, timed: bool = False, stream=None) -> None:
    _check(lib().fft_dist_transform(ctx, _addr(input), _addr(output), direction, int(natural_order), int(timed), _stream(stream)))


def fft_dist_natural_buffer(ctx: int) -> int:
    return lib().fft_dist_natural_buffer(ctx)


def fft_dist_status(ctx: int) -> None:
    _check(lib().fft_dist_status(ctx))


def fft_dist_phase_ms(ctx: int) -> list[float]:
    ms = (C.c_float * 4)()
    _check(lib().fft_dist_phase_ms(ctx, ms))
    return [float(v) for v in ms]


def fft_dist_destroy(ctx: int) -> None:
    lib().fft_dist_destroy(ctx)
