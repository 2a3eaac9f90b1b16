// Host-side launch interface between the plan / C-ABI layer and the kernel translation units.
#pragma once
#include <cuda_runtime.h>

#include "fft_kernels.cuh"
#include "pconv_kernel.cuh"
#include "large_kernels.cuh"
#include "mixed_kernels.cuh"
#include "mixq_kernels.cuh"
#include "cluster_kernels.cuh"

namespace cfb
{
constexpr int kMinLogM = 4;  // 16 complex points per CTA-resident transform
constexpr int kMaxLogM = 14; // 16384 complex points: the largest single-kernel transform
// complex points per thread: 16 everywhere, plus 32 for the sizes where it saves a shared-memory exchange
// (2^9, 2^10, 2^13, 2^14; has_radix32)

// One launch of the single-kernel transform (complex length 2^logM per transform).
// logW: 0 = ordered output/input, 2 / 3 = the reference's 4- / 8-lane unordered layout
cudaError_t launch_fft (int logM, int kind, int logW, int radix, const FftArgs& args, cudaStream_t stream);
bool has_radix32 (int logM);
// the same transform with the conventions of the reference's JUCE adapter (fft_kernel_juce): ordered layouts,
// kind R2C (Nyquist as bin N/2), C2R and C2C_BWD (scaled by 1/N); and the optional negative-frequency mirror
cudaError_t launch_fft_juce (int logM, int kind, int radix, const FftArgs& args, cudaStream_t stream);
cudaError_t launch_juce_mirror (float* data, long long stride, int M, int batch, cudaStream_t stream);
// frame-gather R2C (STFT analysis): transform (o, i) reads in + o in_outer + i in_inner with 0 < in_inner <= N,
// optional window; one CTA gathers the union of its frames once (stft_kernel)
cudaError_t launch_stft (int logM, int logW, int radix, const FftArgs& args, cudaStream_t stream);
// persistent TMA-fed variant (stft_pipe_kernel): needs 0 < in_inner <= N, in_inner % 4 == 0, in_outer % 4 == 0 and a
// 16-byte aligned signal; returns cudaErrorInvalidConfiguration when its buffers do not fit in shared memory
cudaError_t launch_stft_pipe (int logM, int logW, int radix, const FftArgs& args, cudaStream_t stream);
// overlap-add synthesis (istft_kernel): C2R of frames + window + sum at hop distance; args.in_inner / in_outer =
// spectrum frame / channel strides, args.out_inner = hop (0 < hop <= N), args.out_outer = signal channel stride,
// args.inner = frames per channel, args.seg_frames (multiple of transforms_per_cta) and args.nseg = segmentation
cudaError_t launch_istft (int logM, int logW, int radix, const FftArgs& args, cudaStream_t stream);
// overlap-add synthesis with register accumulators (ristft_kernel: complex lengths 2^6 .. 2^12, hq = hop / (2 T) in {2, 4, 8});
// cudaErrorInvalidConfiguration = no such instance.  carry != nullptr: streaming synthesis (ristft_carry_kernel, args.nseg = 1,
// args.seg_frames = args.inner) whose accumulators start from and end in carry, (N - hop) / 2 float2 per channel
cudaError_t launch_ristft (int logM, int hq, int logW, const FftArgs& args, cudaStream_t stream, float2* carry = nullptr);
int transforms_per_cta (int logM, int radix);
// persistent TMA-pipelined variant (pipe_kernels.cuh) for complex lengths 2^13 / 2^14, logW 0 or 3, plain batches
// (args.inner == args.batch) whose input rows are 16-byte aligned
bool has_pipe (int logM);
cudaError_t launch_pipe (int logM, int kind, int logW, const FftArgs& args, cudaStream_t stream);
cudaError_t launch_pipe_13 (int kind, int logW, const FftArgs& args, cudaStream_t stream);
cudaError_t launch_pipe_14 (int kind, int logW, const FftArgs& args, cudaStream_t stream);
// warp-pipelined variant (wpipe_kernel) for the sizes one warp owns (2^10 points with radix 32, 2^9 with radix 16), kinds R2C /
// C2C_FWD, every layout, plain or two-level batches whose input rows are all 16-byte aligned; warps per CTA <= 0 = as
// many as fit one SM
bool has_wpipe (int logM, int radix);
cudaError_t launch_wpipe (int logM, int kind, int logW, int warps, const FftArgs& args, cudaStream_t stream);
cudaError_t launch_wpipe_9 (int kind, int logW, int warps, const FftArgs& args, cudaStream_t stream);
cudaError_t launch_wpipe_10 (int kind, int logW, int warps, const FftArgs& args, cudaStream_t stream);
// warp-pipelined overlap-add synthesis (wistft_kernel) for the same sizes: ordered spectra, hop = N/2, N/4 or N/8
// (hq = hop / 64), 16-byte aligned frames; wistft_warps = warps per CTA (one CTA per SM)
cudaError_t launch_wistft (int logM, int hq, int warps, const FftArgs& args, cudaStream_t stream);
int wistft_warps (int logM);
cudaError_t launch_wistft_9 (int hq, int warps, const FftArgs& args, cudaStream_t stream);
cudaError_t launch_wistft_10 (int hq, int warps, const FftArgs& args, cudaStream_t stream);
int wistft_warps_9();
int wistft_warps_10();
// number of float2 entries of the stage twiddle table for 2^logM, and the fill routine (fp64 -> fp32)
int stage_twiddle_len (int logM, int radix);
void fill_stage_twiddles_rt (int logM, int radix, float2* tw);

// fused partitioned-convolution block step for a REAL plan of 2^(logM+1) samples (one CTA per channel)
cudaError_t launch_pconv (int logM, int logW, const PConvArgs& args, cudaStream_t stream);
// its accumulating modes (streaming convolver): mode PCONV_ADD (with or without a partial spectrum) or PCONV_EMIT; with from_fdl
// (X_t read from the delay line) PCONV_ADD (with or without a partial spectrum) or PCONV_EMIT_MIX
cudaError_t launch_pconv_acc (int logM, int logW, int mode, bool partial, bool from_fdl, const PConvArgs& args, const PConvAcc& acc, cudaStream_t stream);
// the convolver's sliced tail multiply-accumulate, input-history write and IR partition gather (pconv_kernel.cuh)
cudaError_t launch_pconv_slice (const PConvSliceArgs& args, cudaStream_t stream);
cudaError_t launch_conv_input (const ConvInputArgs& args, cudaStream_t stream);
cudaError_t launch_conv_ir_gather (const ConvIrArgs& args, cudaStream_t stream);

// generic mixed-radix transform (N = 2^a 3^b 5^c, not a power of two), one CTA per transform
cudaError_t launch_mixed (const MixedArgs& args, cudaStream_t stream);
// Q x 2^logP transforms (mixq_kernels.cuh); cudaErrorInvalidConfiguration = no such instance
cudaError_t launch_mixq (int logP, int Q, const MixQArgs& args, cudaStream_t stream);

// one-pass cluster transform (cluster_kernels.cuh) for complex lengths 2^15 .. 2^17: plain batches, 16-byte aligned input rows
// with in_stride % 4 == 0; dir < 0 forward (logW 0 or 3 = 8-lane unordered output), dir > 0 backward (logW 0).
// cudaErrorInvalidConfiguration / cudaErrorNotSupported = does not apply (fall back to the multi-pass path)
bool has_cluster (int logN);
cudaError_t launch_cluster_fft (int logN, int dir, int logW, const float* in, long long in_stride, const ClusterArgs& args, cudaStream_t stream);

// multi-pass (large transform) kernels, large_inst.cu
cudaError_t launch_tile (int logL, int C, int dir, bool load_j_fast, int uio, const TileArgs& args, cudaStream_t stream);
struct TilePass; // large_plan.h
// one tile pass through the persistent tensor-map TMA kernel where it applies (tuning hook tile_tma), else tile_fft_kernel
cudaError_t launch_tile_pass (int dir, const TilePass& pass, cudaStream_t stream);
cudaError_t launch_real_pass (int dir, const RealPassArgs& args, int batch, cudaStream_t stream);
cudaError_t launch_dist_barrier (const DistBarrierArgs& args, cudaStream_t stream);

cudaError_t launch_convolve (const float* a, const float* b, float* ab, long long a_stride, long long b_stride, long long ab_stride, int nfloats, int batch, int logW, bool is_real, float scaling, cudaStream_t stream);
cudaError_t launch_accumulate (const float* a, const float* b, float* ab, long long n, cudaStream_t stream);

// every kernel launch made by this library bumps this counter (bench.py reports it as gpu_launches)
unsigned long long launch_count();
void count_launch();
// tuning hook "small": 1 = dense batches of 16 .. 64-point transforms go through the staged kernel (fft_small_kernel), 0 = fft_kernel
int& fft_small_mode();

// per-size entry points, one translation unit each (fft_inst.cu compiled with -DCFB_LOGM=n)
#define CFB_DECL_INST(n)                                                                       \
    cudaError_t launch_fft_##n (int kind, int logW, int radix, const FftArgs& args, cudaStream_t stream); \
    cudaError_t launch_fft_juce_##n (int kind, int radix, const FftArgs& args, cudaStream_t stream); \
    cudaError_t launch_pconv_##n (int logW, const PConvArgs& args, cudaStream_t stream);           \
    cudaError_t launch_pconv_acc_##n (int logW, int mode, bool partial, bool from_fdl, const PConvArgs& args, const PConvAcc& acc, cudaStream_t stream); \
    cudaError_t launch_stft_##n (int logW, int radix, FftArgs args, cudaStream_t stream);          \
    cudaError_t launch_stft_pipe_##n (int logW, int radix, const FftArgs& args, cudaStream_t stream); \
    cudaError_t launch_istft_##n (int logW, int radix, const FftArgs& args, cudaStream_t stream);  \
    cudaError_t launch_ristft_##n (int hq, int logW, const FftArgs& args, cudaStream_t stream, float2* carry); \
    int transforms_per_cta_##n (int radix);                                                    \
    int has_radix32_##n();                                                                     \
    int stage_twiddle_len_##n (int radix);                                                     \
    void fill_stage_twiddles_##n (int radix, float2* tw);
CFB_DECL_INST (4)
CFB_DECL_INST (5)
CFB_DECL_INST (6)
CFB_DECL_INST (7)
CFB_DECL_INST (8)
CFB_DECL_INST (9)
CFB_DECL_INST (10)
CFB_DECL_INST (11)
CFB_DECL_INST (12)
CFB_DECL_INST (13)
CFB_DECL_INST (14)
#undef CFB_DECL_INST
} // namespace cfb
