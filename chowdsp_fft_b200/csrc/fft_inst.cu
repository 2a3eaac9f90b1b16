// Instantiates the single-kernel transform for ONE complex length 2^CFB_LOGM (all kinds, ordered and
// unordered).  Compiled once per size so the sizes build in parallel.
#ifndef CFB_LOGM
#error "compile with -DCFB_LOGM=<4..14>"
#endif
#include <cstdint>

#include "dispatch.h"
#include "pipe_kernels.cuh"

// sizes that also get the 32-points-per-thread geometry (one shared-memory exchange fewer than with 16)
#if CFB_LOGM == 9 || CFB_LOGM == 10 || CFB_LOGM == 13 || CFB_LOGM == 14
#define CFB_HAS_R32 1
#else
#define CFB_HAS_R32 0
#endif

namespace cfb
{
namespace
{
#if CFB_LOGM <= 5
// dense batch of tiny transforms through the staged kernel (fft_small_kernel)?  Rows of 2 M floats on both sides, 8-byte aligned
// bases (16 for the unordered layouts, whose image is drained with 128-bit stores into the shared-memory row anyway)
template <int KIND, int LOGW>
bool small_applies (const FftArgs& a)
{
    using SL = SmallLaunch<CFB_LOGM, KIND, LOGW>;
    constexpr long long ROW = 2LL << CFB_LOGM;
    constexpr uintptr_t AL = LOGW != 0 ? 15 : 7;
    return SL::APPLIES && fft_small_mode() != 0 && a.inner >= a.batch && a.in_inner == ROW && a.out_inner == ROW && a.window == nullptr
           && (reinterpret_cast<uintptr_t> (a.in) & AL) == 0 && (reinterpret_cast<uintptr_t> (a.out) & AL) == 0;
}
template <int KIND, int LOGW>
cudaError_t launch_small (const FftArgs& a, cudaStream_t stream)
{
    using SL = SmallLaunch<CFB_LOGM, KIND, LOGW>;
    using L = Launch<CFB_LOGM, 16>;
    if constexpr (! SL::APPLIES)
        return cudaErrorInvalidConfiguration;
    else
    {
        auto kernel = fft_small_kernel<CFB_LOGM, KIND, LOGW>;
        const cudaError_t e = cudaFuncSetAttribute (kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SL::SMEM_BYTES);
        if (e != cudaSuccess)
            return e;
        if (a.batch <= 0)
            return cudaSuccess;
        const unsigned grid = (unsigned) (((long long) a.batch + L::PER_CTA - 1) / L::PER_CTA);
        kernel<<<grid, L::THREADS, SL::SMEM_BYTES, stream>>> (a);
        count_launch();
        return cudaGetLastError();
    }
}
#endif

template <int R, int KIND, int LOGW>
cudaError_t launch_one (const FftArgs& a, cudaStream_t stream)
{
#if CFB_LOGM <= 5
    if constexpr (R == 16)
        if (small_applies<KIND, LOGW> (a))
            return launch_small<KIND, LOGW> (a, stream);
#endif
    using L = Launch<CFB_LOGM, R>;
    auto kernel = fft_kernel<CFB_LOGM, R, KIND, LOGW>;
    constexpr int smem_bytes = LOGW != 0 ? L::SMEM_BYTES_UNORD : L::SMEM_BYTES;
    if (smem_bytes > 48 * 1024)
    {
        const cudaError_t e = cudaFuncSetAttribute (kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
        if (e != cudaSuccess)
            return e;
    }
    if (a.batch <= 0)
        return cudaSuccess;
    const unsigned grid = (unsigned) (((long long) a.batch + L::PER_CTA - 1) / L::PER_CTA);
    kernel<<<grid, L::THREADS, smem_bytes, stream>>> (a);
    count_launch();
    return cudaGetLastError();
}
} // namespace

#define CFB_CAT2(a, b) a##b
#define CFB_CAT(a, b) CFB_CAT2 (a, b)

// logW: 0 = ordered, 2 = 4-lane unordered layout, 3 = 8-lane unordered layout.  The 8-lane layout needs
// N % 64 == 0 (complex) / N % 128 == 0 (real), i.e. complex length >= 64 here.
namespace
{
template <int R>
cudaError_t launch_fft_r (int kind, int logW, const FftArgs& a, cudaStream_t stream)
{
    switch (kind * 4 + logW)
    {
        case 0: return launch_one<R, C2C_FWD, 0> (a, stream);
        case 2: return launch_one<R, C2C_FWD, 2> (a, stream);
        case 4: return launch_one<R, C2C_BWD, 0> (a, stream);
        case 6: return launch_one<R, C2C_BWD, 2> (a, stream);
        case 8: return launch_one<R, R2C, 0> (a, stream);
        case 10: return launch_one<R, R2C, 2> (a, stream);
        case 12: return launch_one<R, C2R, 0> (a, stream);
        case 14: return launch_one<R, C2R, 2> (a, stream);
#if CFB_LOGM >= 6
        case 3: return launch_one<R, C2C_FWD, 3> (a, stream);
        case 7: return launch_one<R, C2C_BWD, 3> (a, stream);
        case 11: return launch_one<R, R2C, 3> (a, stream);
        case 15: return launch_one<R, C2R, 3> (a, stream);
#endif
        default: return cudaErrorInvalidValue;
    }
}
} // namespace

cudaError_t CFB_CAT (launch_fft_, CFB_LOGM) (int kind, int logW, int radix, const FftArgs& a, cudaStream_t stream)
{
#if CFB_HAS_R32
    if (radix == 32)
        return launch_fft_r<32> (kind, logW, a, stream);
#endif
    return radix == 16 ? launch_fft_r<16> (kind, logW, a, stream) : cudaErrorInvalidValue;
}

namespace
{
template <int R, int KIND>
cudaError_t launch_juce_one (const FftArgs& a, cudaStream_t stream)
{
    using L = Launch<CFB_LOGM, R>;
    auto kernel = fft_kernel_juce<CFB_LOGM, R, KIND>;
    constexpr int smem_bytes = L::SMEM_BYTES;
    if (smem_bytes > 48 * 1024)
    {
        const cudaError_t e = cudaFuncSetAttribute (kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
        if (e != cudaSuccess)
            return e;
    }
    if (a.batch <= 0)
        return cudaSuccess;
    const unsigned grid = (unsigned) (((long long) a.batch + L::PER_CTA - 1) / L::PER_CTA);
    kernel<<<grid, L::THREADS, smem_bytes, stream>>> (a);
    count_launch();
    return cudaGetLastError();
}
template <int R>
cudaError_t launch_juce_r (int kind, const FftArgs& a, cudaStream_t stream)
{
    switch (kind)
    {
        case C2C_BWD: return launch_juce_one<R, C2C_BWD> (a, stream);
        case R2C: return launch_juce_one<R, R2C> (a, stream);
        case C2R: return launch_juce_one<R, C2R> (a, stream);
        default: return cudaErrorInvalidValue;
    }
}
} // namespace

cudaError_t CFB_CAT (launch_fft_juce_, CFB_LOGM) (int kind, int radix, const FftArgs& a, cudaStream_t stream)
{
#if CFB_HAS_R32
    if (radix == 32)
        return launch_juce_r<32> (kind, a, stream);
#endif
    return radix == 16 ? launch_juce_r<16> (kind, a, stream) : cudaErrorInvalidValue;
}

namespace
{
template <int LOGW>
cudaError_t launch_pconv_one (const PConvArgs& a, cudaStream_t stream)
{
    using PL = PConvLaunch<CFB_LOGM>;
    auto kernel = pconv_kernel<CFB_LOGM, LOGW>;
    constexpr int smem_bytes = PL::SMEM_BYTES;
    if (smem_bytes > 48 * 1024)
    {
        const cudaError_t e = cudaFuncSetAttribute (kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
        if (e != cudaSuccess)
            return e;
    }
    if (a.channels <= 0)
        return cudaSuccess;
    kernel<<<(unsigned) ((a.channels + PL::PER_CTA - 1) / PL::PER_CTA), PL::THREADS, smem_bytes, stream>>> (a);
    count_launch();
    return cudaGetLastError();
}
} // namespace

cudaError_t CFB_CAT (launch_pconv_, CFB_LOGM) (int logW, const PConvArgs& a, cudaStream_t stream)
{
    if (logW == 2)
        return launch_pconv_one<2> (a, stream);
#if CFB_LOGM >= 6
    if (logW == 3)
        return launch_pconv_one<3> (a, stream);
#endif
    return cudaErrorInvalidValue;
}

namespace
{
template <int LOGW, int MODE, bool PARTIAL, bool FROM_FDL = false>
cudaError_t launch_pconv_acc_one (const PConvArgs& a, const PConvAcc& x, cudaStream_t stream)
{
    using PL = PConvLaunch<CFB_LOGM>;
    auto kernel = pconv_acc_kernel<CFB_LOGM, LOGW, MODE, PARTIAL, FROM_FDL>;
    constexpr int smem_bytes = PL::SMEM_BYTES;
    if (smem_bytes > 48 * 1024)
    {
        const cudaError_t e = cudaFuncSetAttribute (kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
        if (e != cudaSuccess)
            return e;
    }
    if (a.channels <= 0)
        return cudaSuccess;
    kernel<<<(unsigned) ((a.channels + PL::PER_CTA - 1) / PL::PER_CTA), PL::THREADS, smem_bytes, stream>>> (a, x);
    count_launch();
    return cudaGetLastError();
}
// instances in use: the fused modes, and with FROM_FDL the ones of a second IR bank (ADD, ADD + PARTIAL, EMIT_MIX)
template <int LOGW>
cudaError_t launch_pconv_acc_w (int mode, bool partial, bool from_fdl, const PConvArgs& a, const PConvAcc& x, cudaStream_t stream)
{
    if (from_fdl)
    {
        if (mode == PCONV_EMIT_MIX && ! partial)
            return launch_pconv_acc_one<LOGW, PCONV_EMIT_MIX, false, true> (a, x, stream);
        if (mode == PCONV_ADD)
            return partial ? launch_pconv_acc_one<LOGW, PCONV_ADD, true, true> (a, x, stream) : launch_pconv_acc_one<LOGW, PCONV_ADD, false, true> (a, x, stream);
        return cudaErrorInvalidValue;
    }
    if (mode == PCONV_EMIT && ! partial)
        return launch_pconv_acc_one<LOGW, PCONV_EMIT, false> (a, x, stream);
    if (mode == PCONV_ADD)
        return partial ? launch_pconv_acc_one<LOGW, PCONV_ADD, true> (a, x, stream) : launch_pconv_acc_one<LOGW, PCONV_ADD, false> (a, x, stream);
    return cudaErrorInvalidValue;
}
} // namespace

cudaError_t CFB_CAT (launch_pconv_acc_, CFB_LOGM) (int logW, int mode, bool partial, bool from_fdl, const PConvArgs& a, const PConvAcc& x, cudaStream_t stream)
{
    if (logW == 2)
        return launch_pconv_acc_w<2> (mode, partial, from_fdl, a, x, stream);
#if CFB_LOGM >= 6
    if (logW == 3)
        return launch_pconv_acc_w<3> (mode, partial, from_fdl, a, x, stream);
#endif
    return cudaErrorInvalidValue;
}

namespace
{
template <int R, int LOGW, bool UNION>
cudaError_t launch_stft_one (const FftArgs& a, cudaStream_t stream)
{
    using L = Launch<CFB_LOGM, R>;
    auto kernel = stft_kernel<CFB_LOGM, R, LOGW, UNION>;
    constexpr int smem_bytes = LOGW != 0 ? L::SMEM_BYTES_UNORD : L::SMEM_BYTES;
    static_assert (smem_bytes >= L::PER_CTA * (8 << CFB_LOGM), "the union image must fit in the exchange buffers");
    if (smem_bytes > 48 * 1024)
    {
        const cudaError_t e = cudaFuncSetAttribute (kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
        if (e != cudaSuccess)
            return e;
    }
    if (a.batch <= 0)
        return cudaSuccess;
    const long long outer = a.batch / a.inner;
    kernel<<<(unsigned) (outer * a.groups), L::THREADS, smem_bytes, stream>>> (a);
    count_launch();
    return cudaGetLastError();
}
template <int R>
cudaError_t launch_stft_r (int logW, FftArgs a, cudaStream_t stream)
{
    a.groups = (a.inner + Launch<CFB_LOGM, R>::PER_CTA - 1) / Launch<CFB_LOGM, R>::PER_CTA;
    switch (logW * 2 + (a.union_gather ? 1 : 0))
    {
        case 0: return launch_stft_one<R, 0, false> (a, stream);
        case 1: return launch_stft_one<R, 0, true> (a, stream);
        case 4: return launch_stft_one<R, 2, false> (a, stream);
        case 5: return launch_stft_one<R, 2, true> (a, stream);
#if CFB_LOGM >= 6
        case 6: return launch_stft_one<R, 3, false> (a, stream);
        case 7: return launch_stft_one<R, 3, true> (a, stream);
#endif
        default: return cudaErrorInvalidValue;
    }
}
} // namespace

namespace
{
template <int R, int LOGW>
cudaError_t launch_stft_pipe_one (FftArgs a, cudaStream_t stream)
{
    using SP = StftPipeGeo<CFB_LOGM, R, LOGW>;
    using L = Launch<CFB_LOGM, R>;
    auto kernel = stft_pipe_kernel<CFB_LOGM, R, LOGW>;
    a.groups = (a.inner + L::PER_CTA - 1) / L::PER_CTA;
    a.land_bytes = SP::land_bytes (a.in_inner);
    const int smem_bytes = SP::smem_bytes (a.in_inner);
    if (smem_bytes > 227 * 1024)
        return cudaErrorInvalidConfiguration;
    if (a.batch <= 0)
        return cudaSuccess;
    // resident CTAs for this (device, landing size); the attribute and the occupancy query are cached per thread
    static thread_local int c_dev = -1, c_smem = -1, c_resident = 0;
    int dev = 0;
    cudaError_t e = cudaGetDevice (&dev);
    if (e != cudaSuccess)
        return e;
    if (dev != c_dev || smem_bytes != c_smem)
    {
        int sms = 0, per_sm = 0;
        if ((e = cudaFuncSetAttribute (kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes)) != cudaSuccess
            || (e = cudaDeviceGetAttribute (&sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess
            || (e = cudaOccupancyMaxActiveBlocksPerMultiprocessor (&per_sm, kernel, L::THREADS, (size_t) smem_bytes)) != cudaSuccess)
            return e;
        if (per_sm < 1)
            return cudaErrorInvalidConfiguration;
        c_dev = dev;
        c_smem = smem_bytes;
        c_resident = sms * per_sm;
    }
    const long long items = (long long) (a.batch / a.inner) * a.groups;
    const long long resident = c_resident;
    kernel<<<(unsigned) (items < resident ? items : resident), L::THREADS, smem_bytes, stream>>> (a);
    count_launch();
    return cudaGetLastError();
}
template <int R>
cudaError_t launch_stft_pipe_r (int logW, const FftArgs& a, cudaStream_t stream)
{
    switch (logW)
    {
        case 0: return launch_stft_pipe_one<R, 0> (a, stream);
        case 2: return launch_stft_pipe_one<R, 2> (a, stream);
#if CFB_LOGM >= 6
        case 3: return launch_stft_pipe_one<R, 3> (a, stream);
#endif
        default: return cudaErrorInvalidValue;
    }
}
} // namespace

namespace
{
template <int R, int LOGW>
cudaError_t launch_istft_one (const FftArgs& a, cudaStream_t stream)
{
    using G = Geo<CFB_LOGM, R>;
    using L = Launch<CFB_LOGM, R>;
    auto kernel = istft_kernel<CFB_LOGM, R, LOGW>;
    const int tail_n = 2 * G::M - (int) a.out_inner;
    const int smem_bytes = (LOGW != 0 ? L::SMEM_BYTES_UNORD : L::SMEM_BYTES) + 2 * ((tail_n + 3) & ~3) * 4;
    if (smem_bytes > 227 * 1024)
        return cudaErrorInvalidConfiguration;
    if (smem_bytes > 48 * 1024)
    {
        const cudaError_t e = cudaFuncSetAttribute (kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
        if (e != cudaSuccess)
            return e;
    }
    const long long grid = (long long) (a.batch / a.inner) * a.nseg;
    if (grid <= 0)
        return cudaSuccess;
    kernel<<<(unsigned) grid, L::THREADS, smem_bytes, stream>>> (a);
    count_launch();
    return cudaGetLastError();
}
template <int R>
cudaError_t launch_istft_r (int logW, const FftArgs& a, cudaStream_t stream)
{
    switch (logW)
    {
        case 0: return launch_istft_one<R, 0> (a, stream);
        case 2: return launch_istft_one<R, 2> (a, stream);
#if CFB_LOGM >= 6
        case 3: return launch_istft_one<R, 3> (a, stream);
#endif
        default: return cudaErrorInvalidValue;
    }
}
} // namespace

// overlap-add synthesis with register accumulators (ristft_kernel): hq = hop / (2 T) in {2, 4, 8}; cudaErrorInvalidConfiguration = no such instance.
// carry != nullptr: the streaming variant (ristft_carry_kernel), one item per channel, accumulators loaded from and stored to carry
#if CFB_LOGM >= 6 && CFB_LOGM <= 12
namespace
{
template <int HQ, int LOGW, bool CARRY>
cudaError_t launch_ristft_one (const FftArgs& a, float2* carry, cudaStream_t stream)
{
    using L = Launch<CFB_LOGM, 16>;
    constexpr int smem_bytes = LOGW != 0 ? L::SMEM_BYTES_UNORD : L::SMEM_BYTES;
    if (smem_bytes > 48 * 1024)
    {
        const cudaError_t e = CARRY ? cudaFuncSetAttribute (ristft_carry_kernel<CFB_LOGM, HQ, LOGW>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes)
                                    : cudaFuncSetAttribute (ristft_kernel<CFB_LOGM, HQ, LOGW>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
        if (e != cudaSuccess)
            return e;
    }
    const long long items = (long long) (a.batch / a.inner) * a.nseg;
    if (items <= 0)
        return cudaSuccess;
    const unsigned grid = (unsigned) ((items + L::PER_CTA - 1) / L::PER_CTA);
    if constexpr (CARRY)
        ristft_carry_kernel<CFB_LOGM, HQ, LOGW><<<grid, L::THREADS, smem_bytes, stream>>> (a, carry);
    else
        ristft_kernel<CFB_LOGM, HQ, LOGW><<<grid, L::THREADS, smem_bytes, stream>>> (a);
    count_launch();
    return cudaGetLastError();
}
template <int HQ, bool CARRY>
cudaError_t launch_ristft_h (int logW, const FftArgs& a, float2* carry, cudaStream_t stream)
{
    switch (logW)
    {
        case 0: return launch_ristft_one<HQ, 0, CARRY> (a, carry, stream);
        case 2: return launch_ristft_one<HQ, 2, CARRY> (a, carry, stream);
        case 3: return launch_ristft_one<HQ, 3, CARRY> (a, carry, stream);
        default: return cudaErrorInvalidConfiguration;
    }
}
template <bool CARRY>
cudaError_t launch_ristft_c (int hq, int logW, const FftArgs& a, float2* carry, cudaStream_t stream)
{
    switch (hq)
    {
        case 2: return launch_ristft_h<2, CARRY> (logW, a, carry, stream);
        case 4: return launch_ristft_h<4, CARRY> (logW, a, carry, stream);
        case 8: return launch_ristft_h<8, CARRY> (logW, a, carry, stream);
        default: return cudaErrorInvalidConfiguration;
    }
}
} // namespace
#endif
cudaError_t CFB_CAT (launch_ristft_, CFB_LOGM) (int hq, int logW, const FftArgs& a, cudaStream_t stream, float2* carry)
{
#if CFB_LOGM >= 6 && CFB_LOGM <= 12
    return carry != nullptr ? launch_ristft_c<true> (hq, logW, a, carry, stream) : launch_ristft_c<false> (hq, logW, a, nullptr, stream);
#else
    (void) hq; (void) logW; (void) a; (void) stream; (void) carry;
    return cudaErrorInvalidConfiguration;
#endif
}

// overlap-add synthesis (istft_kernel); a.seg_frames must be a multiple of transforms_per_cta
cudaError_t CFB_CAT (launch_istft_, CFB_LOGM) (int logW, int radix, const FftArgs& a, cudaStream_t stream)
{
#if CFB_HAS_R32
    if (radix == 32)
        return launch_istft_r<32> (logW, a, stream);
#endif
    return radix == 16 ? launch_istft_r<16> (logW, a, stream) : cudaErrorInvalidValue;
}

// persistent TMA-fed frame-gather R2C (stft_pipe_kernel); fills in a.groups and a.land_bytes
cudaError_t CFB_CAT (launch_stft_pipe_, CFB_LOGM) (int logW, int radix, const FftArgs& a, cudaStream_t stream)
{
#if CFB_HAS_R32
    if (radix == 32)
        return launch_stft_pipe_r<32> (logW, a, stream);
#endif
    return radix == 16 ? launch_stft_pipe_r<16> (logW, a, stream) : cudaErrorInvalidValue;
}

// frame-gather R2C (STFT analysis); fills in a.groups
cudaError_t CFB_CAT (launch_stft_, CFB_LOGM) (int logW, int radix, FftArgs a, cudaStream_t stream)
{
#if CFB_HAS_R32
    if (radix == 32)
        return launch_stft_r<32> (logW, a, stream);
#endif
    return radix == 16 ? launch_stft_r<16> (logW, a, stream) : cudaErrorInvalidValue;
}
int CFB_CAT (has_radix32_, CFB_LOGM)() { return CFB_HAS_R32; }
int CFB_CAT (transforms_per_cta_, CFB_LOGM) (int radix)
{
#if CFB_HAS_R32
    if (radix == 32)
        return Launch<CFB_LOGM, 32>::PER_CTA;
#endif
    return Launch<CFB_LOGM, 16>::PER_CTA;
}
int CFB_CAT (stage_twiddle_len_, CFB_LOGM) (int radix)
{
#if CFB_HAS_R32
    if (radix == 32)
        return Geo<CFB_LOGM, 32>::TW_LEN;
#endif
    return Geo<CFB_LOGM, 16>::TW_LEN;
}
void CFB_CAT (fill_stage_twiddles_, CFB_LOGM) (int radix, float2* tw)
{
#if CFB_HAS_R32
    if (radix == 32)
    {
        fill_stage_twiddles<CFB_LOGM, 32> (tw);
        return;
    }
#endif
    fill_stage_twiddles<CFB_LOGM, 16> (tw);
}
} // namespace cfb
