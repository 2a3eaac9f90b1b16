/*
 * B200 extensions to the chowdsp_fft C API: batched, stream-ordered entry points with no analogue in
 * the reference (one reference call = one transform on the calling thread,
 * /root/reference/chowdsp_fft.cpp:318-432).  Semantics of every batched call: bit-for-bit what a loop
 * of `batch` single calls of the matching chowdsp_fft.h function would produce.
 *
 * Plain C ABI: pointers, sizes and an opaque `void* stream` (a cudaStream_t; NULL = the legacy default
 * stream).  All functions return 0 on success or a negative FFT_B200_E* code; fft_b200_last_error()
 * gives the text for the calling thread's last failure.
 *
 * Pointer policy: when every data pointer is device (or managed) memory the call only enqueues work on
 * `stream` and returns.  When the data pointers are host memory the call stages chunks through the
 * device on internal streams (H2D, transform, D2H overlapped) and returns after the result is in the
 * host buffer.  Mixing host and device data pointers in one call is rejected.
 *
 * Streams: `stream` may be NULL, cudaStreamLegacy, cudaStreamPerThread or any created stream, blocking or not; every
 * launch, copy and memset of a call goes to it, and helper streams of the multi-pass schedules are joined back into it
 * before the call returns.  A plan may be used from several threads at once, each on its own stream.
 * CUDA graphs: the stateless device-pointer calls (fft_transform_batched / _strided, fft_stft_forward,
 * fft_istft_overlap_add, fft_juce_*_batched, fft_convolve_unordered_batched, fft_accumulate_batched,
 * fft_partitioned_convolve_step) may be captured (global capture mode) and replayed, with no eager warm-up, from any
 * thread: setup uploads the tables and sets the device memory pool's release threshold, so a call makes no
 * capture-illegal API call.  Exception: the first call of a plan on a device other than the one it was created on
 * builds that device's tables with blocking allocations; make it eagerly.  The streaming contexts (fft_convolver_*,
 * fft_stft_stream_*) keep their block / frame counts on the host, so a replayed capture would repeat one block: they
 * are not replayable.
 * tests/test_gpu_streams.py checks all of this against float64 and against calls on the default stream.
 */
#pragma once
#include "chowdsp_fft.h"

#ifdef __cplusplus
extern "C"
{
namespace chowdsp::fft
{
#endif

enum
{
    FFT_B200_OK = 0,
    FFT_B200_EINVAL = -1,   /* bad handle / argument */
    FFT_B200_ECUDA = -2,    /* CUDA runtime error, see fft_b200_last_error() */
    FFT_B200_ENODEVICE = -3 /* no usable CUDA device: there is no CPU fallback */
};

/* `batch` transforms; transform b reads input + b*in_stride and writes output + b*out_stride (strides in
   floats).  ordered != 0 behaves like fft_transform, 0 like fft_transform_unordered.
   Replaces a loop over reference chowdsp_fft.h:138 / :145. */
int fft_transform_batched (void* setup, const float* input, float* output, int batch, long long in_stride, long long out_stride, fft_direction_t direction, int ordered, void* stream);

/* Two-level batch: transform (o, i), o < outer, i < inner, reads input + o*in_outer + i*in_inner and
   writes output + o*out_outer + i*out_inner.  Input windows may overlap (STFT frame gather:
   in_inner = hop, in_outer = channel stride); outputs must not.  Device pointers: stream-ordered.  Host pointers (both
   buffers; the reference API is host-pointer only): synchronous, the UNIQUE input span of every outer index crosses PCIe
   once, in chunks overlapped with the kernels and the downloads (needs in_inner >= 0 and in_outer >= that span). */
int fft_transform_strided (void* setup, const float* input, float* output, int outer, int inner, long long in_outer, long long in_inner, long long out_outer, long long out_inner, fft_direction_t direction, int ordered, void* stream);

/* Short-time Fourier analysis of `channels` real signals: frame f of channel c is the N samples at
   signal + c*channel_stride + f*hop (0 < hop, frames may overlap), multiplied by window[0..N) when window
   is non-NULL (NULL = rectangular, which is what a loop over reference chowdsp_fft.h:138 computes), and its
   forward real transform is written to spectra + c*out_channel_stride + f*out_frame_stride (N floats,
   ordered pffft packing or the unordered layout).  One kernel, the window multiply is fused into the load.
   hop and channel_stride must be even.  Device pointers: stream-ordered.  Host pointers (signal and spectra; the window
   may live on either side): synchronous, every channel's samples are uploaded once -- not once per overlapping frame. */
int fft_stft_forward (void* setup, const float* signal, float* spectra, int channels, int frames, long long channel_stride, long long hop, long long out_channel_stride, long long out_frame_stride, const float* window, int ordered, void* stream);

/* Overlap-add synthesis (inverse STFT) of `channels` signals from `frames` spectra each: the backward real transform
   of the spectrum at spectra + c*spec_channel_stride + f*spec_frame_stride (N floats, ordered pffft packing or the
   plan's unordered layout) is multiplied by scale and by window[0..N) when window is non-NULL, and added into
   signal + c*channel_stride at offset f*hop.  Every one of the (frames-1)*hop + N output samples of a channel is
   WRITTEN (the sum of the frames covering it), so the buffer needs no clearing.  Unnormalised like the reference:
   scale = 1/N undoes fft_stft_forward for a rectangular window at hop = N.  This is the step the reference leaves
   to its callers around fft_transform (BACKWARD) and fft_accumulate (chowdsp_fft.h:138,160); here it is one kernel,
   owner-computes (no atomics, bit-reproducible).  0 < hop <= N, even spectrum strides, N <= 16384.  Device pointers:
   stream-ordered.  Host pointers (spectra and signal): synchronous, staged in chunks of channels. */
int fft_istft_overlap_add (void* setup, const float* spectra, float* signal, int channels, int frames, long long spec_channel_stride, long long spec_frame_stride, long long channel_stride, long long hop, const float* window, float scale, int ordered, void* stream);

/* The conventions of the reference's JUCE adapter (chowdsp_fft_juce/chowdsp_fft_juce.cpp:32-86), batched and fused
   into the transform kernels' loads and stores.  Power-of-two plans up to the single-kernel limit, device pointers,
   even strides.
     fft_juce_perform_batched       juce::dsp::FFT::perform: complex, interleaved; inverse != 0 scales by 1/N
     fft_juce_real_forward_batched  performRealOnlyForwardTransform: every row holds 2 N floats (N + 2 suffice when
                                    ignore_negative_freqs != 0); N real samples in, N/2 + 1 interleaved complex bins
                                    out (Im of DC and of Nyquist = 0), plus -- unless ignore_negative_freqs -- the
                                    conjugate mirror in bins N/2+1 .. N-1
     fft_juce_real_inverse_batched  performRealOnlyInverseTransform: N/2 + 1 interleaved bins in, N real samples out,
                                    scaled by 1/N
   In place, like the JUCE interface (row b at inout + b * stride floats). */
int fft_juce_perform_batched (void* setup_complex, const float* input, float* output, int batch, long long in_stride, long long out_stride, int inverse, void* stream);
int fft_juce_real_forward_batched (void* setup_real, float* inout, int batch, long long stride, int ignore_negative_freqs, void* stream);
int fft_juce_real_inverse_batched (void* setup_real, float* inout, int batch, long long stride, void* stream);

/* batch x (ab += a*b*scaling) on unordered spectra; a stride of 0 shares that operand across the
   batch (e.g. one impulse response for all channels).  Replaces a loop over reference chowdsp_fft.h:154. */
int fft_convolve_unordered_batched (void* setup, const float* dft_a, const float* dft_b, float* dft_ab, int batch, long long a_stride, long long b_stride, long long ab_stride, float scaling, void* stream);

/* One block step of a uniform partitioned overlap-save convolution ("convolution reverb") for `channels`
   independent channels, fused into a single kernel.  setup must be a REAL plan of size N; B = N/2 new
   samples per block; every spectrum is in the plan's unordered layout.  Per channel c:
     X        = fft_transform_unordered (FORWARD) of the N samples at windows + c*window_stride
                (previous block followed by the new block)
     fdl slot = fdl + c*fdl_channel_stride + (block_index % partitions)*N   <- X   (frequency-delay line)
     Y        = sum over p = 0 .. min(block_index, partitions-1) of
                  fdl[c][(block_index - p) % partitions] * ir[c][p] * scaling      (fft_convolve_unordered)
                with ir[c][p] at ir + c*ir_channel_stride + p*N  (ir_channel_stride = 0: one IR for all)
     output + c*output_stride  <- last B samples of fft_transform_unordered (BACKWARD) of Y
   i.e. exactly the reference sequence chowdsp_fft.h:145 ; partitions x :154 ; :145 per channel and block
   (test/test.cpp:214-218 shows the pattern), in one launch.  Device pointers only; stream-ordered. */
int fft_partitioned_convolve_step (void* setup, const float* windows, long long window_stride, const float* ir, long long ir_channel_stride, float* fdl, long long fdl_channel_stride, float* output, long long output_stride, int channels, int partitions, int block_index, float scaling, void* stream);

/* Streaming convolution of `channels` real signals with long impulse responses at a small block size: a stateful context
   that takes B = block_size new samples per channel per call and returns B convolved samples per channel, with no added
   latency.  Call t (counted from create or reset) reads x_c[tB .. (t+1)B) at input + c*input_stride and writes
   y_c[tB .. (t+1)B) at output + c*output_stride, where y_c[n] = sum_{m < ir_length} h_c[m] x_c[n-m] (the true linear
   convolution, normalised; the input before the first call is silence).  h_c is at ir + c*ir_channel_stride;
   ir_channel_stride = 0 shares one IR across all channels (stored and transformed once).
   The IR is split non-uniformly (fft_convolver_segments reports the schedule): segment 0 has block B and two partitions,
   segment k >= 1 block 2^k B and one partition, up to the largest block Bmax (16384, tuning hook "convolver_max_block"),
   which takes the rest of the IR; small blocks keep the latency, large ones cut the memory traffic per sample.
     fft_convolver_create    allocates and zeroes the state and transforms the IR partitions (synchronous on `stream`);
                             16 <= block_size <= 16384, a power of two; ir_length >= 1; ir_channel_stride 0 or >= ir_length
     fft_convolver_process   one block per channel; input / output 8-byte aligned with even strides; stream-ordered
     fft_convolver_set_ir    replaces the IR on a live context, instantly or with a crossfade (below); stream-ordered
     fft_convolver_reset     back to silence (the newest IR is kept, a running crossfade ends); stream-ordered
     fft_convolver_segments  up to max_segments (block size, partitions) pairs (either array may be NULL); returns the count
     fft_convolver_destroy   waits for the device, then frees the context (both IR banks)
   Device pointers only.  Calls on one context must be ordered on one stream, on the device that was current at create,
   and a context must not be used from two threads at the same time.

   fft_convolver_set_ir (ctx, ir, ir_length, ir_channel_stride, fade_blocks, stream): switches to the IR h' at ir (layout as
   at create) while audio runs, without cutting the reverb tail of what was already played.  With t0 the number of process
   calls since create / reset, call t >= t0 writes
       y[n] = (1 - g[n]) (h * x)[n] + g[n] (h' * x)[n],   g[n] = min((n - t0 B + 1) / (fade_blocks B), 1),
   both convolutions over the whole input history; fade_blocks = 0 switches at once (g = 1 from call t0 on).  Once the fade
   is over, every output is bit-identical to that of a context created with h' (zero-padded to the create-time length) and
   fed the same input from its first call.  1 <= ir_length <= the ir_length given at create (the schedule is fixed; a
   shorter IR is zero-padded); ir_channel_stride 0 for a context created with a shared IR, else >= ir_length; 4-byte aligned
   device pointer; fade_blocks >= 0 with fade_blocks * B <= 2^24.  During a fade every process call runs both IRs (about
   twice the work); a call while a fade is running, or with a bad argument, returns FFT_B200_EINVAL and leaves the context
   unchanged.  Stream-ordered: ir is read when `stream` reaches the call.  The first call on a context allocates the second
   IR bank and a gather buffer and may synchronise, like create; to keep that off an audio thread, call it once at start-up
   with the current IR (fade_blocks = 0).  Every later call allocates nothing and does not block the host. */
int fft_convolver_create (int channels, int block_size, const float* ir, long long ir_length, long long ir_channel_stride, void* stream, void** ctx_out);
int fft_convolver_process (void* ctx, const float* input, long long input_stride, float* output, long long output_stride, void* stream);
int fft_convolver_set_ir (void* ctx, const float* ir, long long ir_length, long long ir_channel_stride, int fade_blocks, void* stream);
int fft_convolver_reset (void* ctx, void* stream);
int fft_convolver_segments (void* ctx, int* block_sizes, int* partitions, int max_segments);
int fft_convolver_destroy (void* ctx);

/* Streaming STFT of `channels` real signals for real-time spectral processing (denoisers, spectral gates, vocoders): a stateful
   context that turns hop new samples per channel into one spectrum (analysis), and one spectrum into hop finished samples
   (overlap-add synthesis), `frames` at a time, keeping its own input history and overlap-add tail.
     fft_stft_stream_create      setup: a REAL power-of-two plan with 128 <= N <= 8192 (the context keeps its own copy; the setup
                                 may be destroyed afterwards); hop = N/2, N/4 or N/8; 1 <= frames <= max_frames on every call.
                                 The windows (N floats, host or device, NULL = rectangular) are copied: the caller may free them
                                 when create returns.  Spectra in the plan's ordered (ordered != 0) or unordered layout,
                                 synthesis scaled by `scale`.  Allocates and zeroes all state; synchronous on `stream`.
     fft_stft_stream_analyze     consumes frames * hop samples per channel at input + c*input_stride (8-byte aligned, even
                                 stride) and writes `frames` spectra at spectra + c*spec_channel_stride + f*spec_frame_stride
     fft_stft_stream_synthesize  reads `frames` spectra (same layout) and writes frames * hop samples per channel at
                                 output + c*output_stride (8-byte aligned, even stride)
     fft_stft_stream_reset       back to silence: both frame counts to zero
     fft_stft_stream_destroy     waits for the device, then frees the context
   Analysis: with x_c the samples passed to analyze for channel c since create / reset, preceded by N - hop zeros, the j-th
   spectrum is frame j of fft_stft_forward on x_c: the forward transform of analysis_window * x_c[j hop, j hop + N), bit for bit.
   Synthesis: with S_j the j-th spectrum passed to synthesize since create / reset, the concatenated output is the first J hop
   samples of fft_istft_overlap_add (S_0 .. S_{J-1}, hop, synthesis_window, scale) -- the samples no later frame reaches --
   bit-identical however the frames are split into calls.  Analysis followed by synthesis returns the input delayed by N - hop,
   scaled by the window-overlap sum.  The two directions keep independent frame counts; a context may be used for one only.
   Spectrum alignment as for fft_istft_overlap_add (8-byte, 16-byte for unordered spectra).  Device pointers only; analyze,
   synthesize and reset are stream-ordered, allocate nothing and do not block the host.  Calls on one context must be ordered
   on one stream, on the device that was current at create, and a context must not be used from two threads at the same time.
   A bad argument returns FFT_B200_EINVAL and leaves the context unchanged. */
int fft_stft_stream_create (void* setup, int channels, long long hop, int max_frames, const float* analysis_window, const float* synthesis_window, float scale,
                            int ordered, void* stream, void** ctx_out);
int fft_stft_stream_analyze (void* ctx, const float* input, long long input_stride, int frames, float* spectra, long long spec_channel_stride, long long spec_frame_stride, void* stream);
int fft_stft_stream_synthesize (void* ctx, const float* spectra, long long spec_channel_stride, long long spec_frame_stride, int frames, float* output, long long output_stride, void* stream);
int fft_stft_stream_reset (void* ctx, void* stream);
int fft_stft_stream_destroy (void* ctx);

/* Distributed four-step transform of ONE complex transform of N = 2^n >= 2^21 points over `world` GPUs
   (one process per GPU): the three LOCAL phases; the exchange between phase 0 and phase 1 is an
   all-to-all of equal contiguous chunks (NCCL, or peer stores, see fft_dist_phase0_peer).
   With N = L1*L2*L3 (fft_large_factors) and S1 = L2*L3, in complex elements:
     phase 0  in : this rank's column block  A[n1][c] = x[n1*S1 + rank*S1/world + c]   ([L1][S1/world])
              out: same shape; row block h (rows h*L1/world ...) is the contiguous chunk for rank h
     phase 1  in : exchange layout [world][L1/world][S1/world] (chunk g came from rank g)
              out: natural rows [L1/world][S1]
     phase 2  in : phase 1's output ; out: "transposed-out" [S1][L1/world],
              out[q][k] = X[(rank*L1/world + k) + L1*q]   (direction FFT_FORWARD; BACKWARD is the conjugate)
   world must be a power of two with L1/world >= 8.  Device pointers, stream-ordered. */
int fft_dist_phase (void* setup, int phase, int rank, int world, const float* in, float* out, fft_direction_t direction, void* stream);

/* Phase 0 fused with the exchange: same input contract as fft_dist_phase (phase 0), but every output row block is
   stored straight into its owner's phase-1 input buffer -- peer_recv[h] is rank h's exchange-layout buffer
   ([world][L1/world][S1/world] complex) mapped into this process (peer memory over NVLink; peer_recv[rank] is
   this rank's own buffer).  The all-to-all is done by the kernel's stores and overlaps its butterflies; the
   caller only needs a barrier across ranks before phase 1 reads the buffers.  world <= 8. */
int fft_dist_phase0_peer (void* setup, int rank, int world, const float* in, float* const* peer_recv, fft_direction_t direction, void* stream);

/* Peer-memory plumbing for fft_dist_phase0_peer, one process per GPU: device blocks that can be exported to the
   other ranks (64-byte opaque IPC handle, exchanged by the caller, e.g. over torch.distributed) and mapped there. */
void* fft_dist_alloc (size_t bytes);
void fft_dist_free (void* block);
int fft_dist_ipc_export (void* block, void* handle64);
void* fft_dist_ipc_open (const void* handle64);
void fft_dist_ipc_close (void* mapped);

/* The distributed transform as ONE call per rank (one process per GPU; SURVEY.md §8e): the reference's contract is a single
   fft_transform call (chowdsp_fft.cpp:318-356), so the exchange orchestration lives behind the C ABI and needs no
   collective library -- the all-to-all is done by the phase-0 kernel's peer stores over NVLink, the barrier across ranks
   is a flag exchange in peer memory executed in the caller's stream, and phases 1 + 2 run L2-chunked.
     fft_dist_create     allocates this rank's two exchange buffers, its natural-order block and its barrier flags
     fft_dist_export     writes fft_dist_blob_bytes() opaque bytes (CUDA IPC handles) that the caller ships to every
                         other rank over any transport (MPI, torch.distributed, files ...) -- like a communicator id
     fft_dist_connect    takes all ranks' blobs, rank-major (blob of rank r at offset r * fft_dist_blob_bytes()), and maps
                         the peers' buffers; world == 1 needs no blobs
     fft_dist_transform  input : this rank's column block  A[n1][c] = x[n1*S1 + rank*S1/world + c]  ([L1][S1/world] complex)
                         natural_order = 0: output = transposed-out [S1][L1/world], out[q][k] = X[(rank*L1/world + k) + L1*q]
                         natural_order = 1: the second all-to-all is fused into the last pass's peer stores; this rank's
                                            contiguous block X[rank*N/world, (rank+1)*N/world) lands in
                                            fft_dist_natural_buffer() and is copied to `output` unless output is that
                                            buffer or NULL
                         timed != 0: records events around the phases and blocks until done; fft_dist_phase_ms then
                                     returns { phase 0 incl. peer stores, barrier wait, phases 1+2, natural barrier + copy }
                         Collective: every rank must call it the same number of times.  A peer that never arrives makes
                         the in-stream barrier give up after 20 s and raises fft_dist_status() instead of hanging the GPU.
   world <= 8, power of two, L1/world >= 16.  Device pointers, stream-ordered. */
int fft_dist_create (void* setup, int rank, int world, void** ctx_out);
size_t fft_dist_blob_bytes (void);
int fft_dist_export (void* ctx, void* blob);
int fft_dist_connect (void* ctx, const void* blobs);
int fft_dist_transform (void* ctx, const float* input, float* output, fft_direction_t direction, int natural_order, int timed, void* stream);
float* fft_dist_natural_buffer (void* ctx);
int fft_dist_status (void* ctx);
int fft_dist_phase_ms (void* ctx, float* ms4);
int fft_dist_destroy (void* ctx);

/* log2 of the pass lengths of a multi-pass plan (l2 = 0 for two-pass plans); returns FFT_B200_EINVAL for
   single-kernel plans. */
int fft_large_factors (void* setup, int* l1, int* l2, int* l3);

/* ab[i] = a[i] + b[i] for n floats (n % 8 == 0), stream-ordered.  Reference chowdsp_fft.h:160. */
int fft_accumulate_batched (void* setup, const float* a, const float* b, float* ab, long long n, void* stream);

/* Text of the calling thread's most recent failure ("" if none), and a way to reset it (the
   reference-shaped functions return void, so callers that want to detect failures clear, call, read). */
const char* fft_b200_last_error (void);
void fft_b200_clear_error (void);

/* Tuning hook for benchmarks / A-B sweeps (not needed in normal use; value -1 restores a key's built-in default where one exists):
     "radix32_mask" bit n (complex plans) / bit 16+n (real plans): 32 points per thread for complex length 2^n (n in 9, 10, 13, 14)
     "pipe_mask"    which kinds / layouts at complex length 2^13, 2^14 use the persistent TMA-pipelined kernel
     "wpipe"        bit 1: overlapping / windowed frames of N = 2048 real transforms use the warp-pipelined kernel (default), bit 3: those of
                    N = 1024 too (measured 8..11 % slower), bit 0: every batch of those sizes; bits 8..: warps per CTA (0 = as many as fit)
     "wistft"       bit 0: overlap-add synthesis of ordered N = 2048 frames through the warp-pipelined kernel (default), bit 1: N = 1024 too;
                    bits 8..: warps per CTA
     "stft_pipe", "stft_union"  older frame-gather variants (persistent CTA-level TMA union / LDS-STS union staging), off
     "tile_c", "tile_c_jfast"   transforms per tile of the multi-pass kernels (8, 16, or 0 = built-in policy)
     "spin_sync"    1 = small synchronous drop-in calls wait on a stream-written word in mapped memory instead of
                    cudaStreamSynchronize; default 0 (measured 1.4 us slower per call on B200)
     "cluster"      1 = complex transforms of 2^15 .. 2^17 points run in one pass on a thread-block cluster (csrc/cluster_kernels.cuh),
                    0 = two tile passes (default: the cluster kernel measured 5..30 % slower); bit 1 (value 3) = without the
                    tensor-map L2 prefetch; "cluster_min_batch": smaller batches stay with the tile passes (default 8)
     "l2_chunk_mb"  MiB of intermediate per chunk of the L2-chunked multi-pass schedules (default 16, applied up to 2^24 points;
                    0 = whole-array passes everywhere; -m (m >= 2) = m MiB chunks at every size)
     "l2_lanes"     helper streams / ring slots the chunks alternate over (1..4, default 3)
     "l2_policy"    1 = evict_last / evict_first L2 hints on ring / streaming accesses of the chunked schedules (default)
     "tile_pf"      tensor-map L2 prefetch distance of the multi-pass tile kernels in tiles (default 0 = off: measured 3..10 % slower)
     "ristft"       1 = overlap-add synthesis with hop = N/2, N/4, N/8 at N = 1024 .. 8192 keeps its sums in registers (ristft_kernel; default),
                    0 = istft_kernel (shared-memory frame buffers and carried tails)
     "small"        1 = dense batches of 16- / 32-point complex transforms run in the staged fft_small_kernel (default), 0 = fft_kernel
     "mixq"         1 = sizes Q 2^p with Q in {3, 5, 9, 15} run in mixq_kernel (default), 0 = always the generic mixed-radix kernel
     "zero_copy_kb" pinned (device-mapped) host buffers up to this many KiB are transformed in place over PCIe by the kernel's own
                    loads / stores instead of being staged through device memory (default 256)
     "pf_ahead"     L2 prefetch distance of the single-kernel transforms in CTAs (default 0 = off)
     "convolver_max_block"  largest block of the streaming convolver's schedule for contexts created afterwards: a power of two
                    in [16, 16384] (default 16384; a value <= block_size makes the schedule uniform) */
int fft_b200_set_tuning (const char* key, int value);

/* Number of CUDA kernels this library has launched in this process (all threads). */
unsigned long long fft_b200_launch_count (void);
/* Name (template instance) of the transform kernel the calling thread launched last, "" if none yet: which of the
 * kernels in csrc/ a given size / kind / layout / alignment was routed to.  Diagnostic only (bench.py reports it). */
const char* fft_b200_last_kernel (void);

/* 1 if a CUDA device is usable from this process, else 0. */
int fft_b200_device_available (void);

#ifdef __cplusplus
}
} // namespace chowdsp::fft
#endif
