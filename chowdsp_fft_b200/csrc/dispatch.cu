// Runtime size dispatch + the elementwise (unordered-domain) kernels.
#include <atomic>

#include "dispatch.h"
#include "elementwise_kernels.cuh"

namespace cfb
{
namespace
{
std::atomic<unsigned long long> g_launches { 0 };
}
static int elementwise_grid (long long items, int threads);
unsigned long long launch_count() { return g_launches.load (std::memory_order_relaxed); }
void count_launch() { g_launches.fetch_add (1, std::memory_order_relaxed); }

#define CFB_FOR_SIZES(X) X (4) X (5) X (6) X (7) X (8) X (9) X (10) X (11) X (12) X (13) X (14)

cudaError_t launch_fft (int logM, int kind, int logW, int radix, const FftArgs& args, cudaStream_t stream)
{
    switch (logM)
    {
#define X(n) \
    case n: return launch_fft_##n (kind, logW, radix, args, stream);
        CFB_FOR_SIZES (X)
#undef X
        default: return cudaErrorInvalidValue;
    }
}
cudaError_t launch_pconv (int logM, int logW, const PConvArgs& args, cudaStream_t stream)
{
    switch (logM)
    {
#define X(n) \
    case n: return launch_pconv_##n (logW, args, stream);
        CFB_FOR_SIZES (X)
#undef X
        default: return cudaErrorInvalidValue;
    }
}
cudaError_t launch_pconv_acc (int logM, int logW, int mode, bool partial, bool from_fdl, const PConvArgs& args, const PConvAcc& acc, cudaStream_t stream)
{
    switch (logM)
    {
#define X(n) \
    case n: return launch_pconv_acc_##n (logW, mode, partial, from_fdl, args, acc, stream);
        CFB_FOR_SIZES (X)
#undef X
        default: return cudaErrorInvalidValue;
    }
}
cudaError_t launch_pconv_slice (const PConvSliceArgs& args, cudaStream_t stream)
{
    const long long items = (long long) args.channels * args.pairs;
    if (items <= 0)
        return cudaSuccess;
    pconv_slice_kernel<<<(unsigned) ((items + 255) / 256), 256, 0, stream>>> (args);
    count_launch();
    return cudaGetLastError();
}
cudaError_t launch_conv_input (const ConvInputArgs& args, cudaStream_t stream)
{
    const long long items = (long long) args.channels * args.half_block;
    if (items <= 0)
        return cudaSuccess;
    conv_input_kernel<<<(unsigned) ((items + 255) / 256), 256, 0, stream>>> (args);
    count_launch();
    return cudaGetLastError();
}
cudaError_t launch_conv_ir_gather (const ConvIrArgs& args, cudaStream_t stream)
{
    const long long items = (long long) args.channels * args.P * 2 * args.Bk;
    if (items <= 0)
        return cudaSuccess;
    conv_ir_gather_kernel<<<elementwise_grid (items, 256), 256, 0, stream>>> (args);
    count_launch();
    return cudaGetLastError();
}
cudaError_t launch_fft_juce (int logM, int kind, int radix, const FftArgs& args, cudaStream_t stream)
{
    switch (logM)
    {
#define X(n) \
    case n: return launch_fft_juce_##n (kind, radix, args, stream);
        CFB_FOR_SIZES (X)
#undef X
        default: return cudaErrorInvalidValue;
    }
}
bool has_pipe (int logM) { return logM == 13 || logM == 14; }
cudaError_t launch_wistft (int logM, int hq, int warps, const FftArgs& args, cudaStream_t stream)
{
    switch (logM)
    {
        case 9: return launch_wistft_9 (hq, warps, args, stream);
        case 10: return launch_wistft_10 (hq, warps, args, stream);
        default: return cudaErrorInvalidValue;
    }
}
int wistft_warps (int logM) { return logM == 9 ? wistft_warps_9() : logM == 10 ? wistft_warps_10() : 0; }
bool has_wpipe (int logM, int radix) { return (logM == 10 && radix == 32) || (logM == 9 && radix == 16); }
cudaError_t launch_wpipe (int logM, int kind, int logW, int warps, const FftArgs& args, cudaStream_t stream)
{
    switch (logM)
    {
        case 9: return launch_wpipe_9 (kind, logW, warps, args, stream);
        case 10: return launch_wpipe_10 (kind, logW, warps, args, stream);
        default: return cudaErrorInvalidValue;
    }
}
cudaError_t launch_pipe (int logM, int kind, int logW, const FftArgs& args, cudaStream_t stream)
{
    switch (logM)
    {
        case 13: return launch_pipe_13 (kind, logW, args, stream);
        case 14: return launch_pipe_14 (kind, logW, args, stream);
        default: return cudaErrorInvalidValue;
    }
}
bool has_radix32 (int logM)
{
    switch (logM)
    {
#define X(n) \
    case n: return has_radix32_##n() != 0;
        CFB_FOR_SIZES (X)
#undef X
        default: return false;
    }
}
cudaError_t launch_stft (int logM, int logW, int radix, const FftArgs& args, cudaStream_t stream)
{
    switch (logM)
    {
#define X(n) \
    case n: return launch_stft_##n (logW, radix, args, stream);
        CFB_FOR_SIZES (X)
#undef X
        default: return cudaErrorInvalidValue;
    }
}
cudaError_t launch_stft_pipe (int logM, int logW, int radix, const FftArgs& args, cudaStream_t stream)
{
    switch (logM)
    {
#define X(n) \
    case n: return launch_stft_pipe_##n (logW, radix, args, stream);
        CFB_FOR_SIZES (X)
#undef X
        default: return cudaErrorInvalidValue;
    }
}
cudaError_t launch_ristft (int logM, int hq, int logW, const FftArgs& args, cudaStream_t stream, float2* carry)
{
    switch (logM)
    {
#define X(n) \
    case n: return launch_ristft_##n (hq, logW, args, stream, carry);
        CFB_FOR_SIZES (X)
#undef X
        default: return cudaErrorInvalidConfiguration;
    }
}
cudaError_t launch_istft (int logM, int logW, int radix, const FftArgs& args, cudaStream_t stream)
{
    switch (logM)
    {
#define X(n) \
    case n: return launch_istft_##n (logW, radix, args, stream);
        CFB_FOR_SIZES (X)
#undef X
        default: return cudaErrorInvalidValue;
    }
}
int transforms_per_cta (int logM, int radix)
{
    switch (logM)
    {
#define X(n) \
    case n: return transforms_per_cta_##n (radix);
        CFB_FOR_SIZES (X)
#undef X
        default: return 1;
    }
}
int stage_twiddle_len (int logM, int radix)
{
    switch (logM)
    {
#define X(n) \
    case n: return stage_twiddle_len_##n (radix);
        CFB_FOR_SIZES (X)
#undef X
        default: return -1;
    }
}
void fill_stage_twiddles_rt (int logM, int radix, float2* tw)
{
    switch (logM)
    {
#define X(n) \
    case n: fill_stage_twiddles_##n (radix, tw); return;
        CFB_FOR_SIZES (X)
#undef X
        default: return;
    }
}

int& fft_small_mode()
{
    static int v = 1;
    return v;
}

cudaError_t launch_mixed (const MixedArgs& args, cudaStream_t stream)
{
    MixedArgs a = args;
    if (a.M > kMixedMaxM || a.nstages <= 0)
        return cudaErrorInvalidValue;
    int threads = 0;
    mixed_geometry (a.M, threads, a.tg);
    const int per_cta = threads / a.tg;
    const int smem_bytes = 16 * a.M * per_cta;
    if (smem_bytes > 48 * 1024)
    {
        const cudaError_t e = cudaFuncSetAttribute (mixed_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
        if (e != cudaSuccess)
            return e;
    }
    if (a.batch <= 0)
        return cudaSuccess;
    const long long ctas = ((long long) a.batch + per_cta - 1) / per_cta, cap = 148LL * 16;
    mixed_kernel<0><<<(unsigned) (ctas < cap ? ctas : cap), threads, smem_bytes, stream>>> (a);
    count_launch();
    return cudaGetLastError();
}

static int elementwise_grid (long long items, int threads)
{
    // enough CTAs to fill 148 SMs x 8 resident CTAs, grid-stride beyond that
    const long long want = (items + threads - 1) / threads;
    const long long cap = 148LL * 8 * 4;
    return (int) (want < 1 ? 1 : (want > cap ? cap : want));
}

cudaError_t launch_convolve (const float* a, const float* b, float* ab, long long a_stride, long long b_stride, long long ab_stride, int nfloats, int batch, int logW, bool is_real, float scaling, cudaStream_t stream)
{
    if (batch <= 0)
        return cudaSuccess;
    const ConvArgs p { a, b, ab, a_stride, b_stride, ab_stride, nfloats, batch, logW, is_real ? 1 : 0, scaling };
    const long long items = (long long) (nfloats >> 3) * batch;
    convolve_kernel<<<elementwise_grid (items, 256), 256, 0, stream>>> (p);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_juce_mirror (float* data, long long stride, int M, int batch, cudaStream_t stream)
{
    const long long total = (long long) batch * (M - 1);
    if (total <= 0)
        return cudaSuccess;
    juce_mirror_kernel<<<elementwise_grid (total, 256), 256, 0, stream>>> (data, stride, M, total);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_accumulate (const float* a, const float* b, float* ab, long long n, cudaStream_t stream)
{
    if (n <= 0)
        return cudaSuccess;
    accumulate_kernel<<<elementwise_grid (n / 4, 256), 256, 0, stream>>> (a, b, ab, n / 4);
    count_launch();
    return cudaGetLastError();
}
} // namespace cfb
