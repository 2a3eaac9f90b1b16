// TEST INFRASTRUCTURE ONLY -- the streaming convolver's kernels (pconv_kernel.cuh, elementwise_kernels.cuh) run on the host
// through cuda_emu.h, like emu_driver.cpp does for the other kernels.  Built into its own library by tests/test_emu_convolver.py;
// not part of the product, never loaded by the package.
#define CHOWDSP_EMU 1
#include "fft_kernels.cuh"
#include "elementwise_kernels.cuh"
#include "pconv_kernel.cuh"

using namespace cfb;

extern "C"
{
// the streaming convolver's accumulating modes of the same step: mode 1 = PCONV_ADD, 2 = PCONV_EMIT; S != nullptr = PARTIAL
int emu_pconv_acc (int logM, int logW, int mode, const float* in, long long in_stride, const float* ir, long long ir_ch_stride, float* fdl, long long fdl_ch_stride,
                   float* out, long long out_stride, float* acc, long long acc_stride, const float* S, long long s_stride, int channels, int P, int t, float scaling)
{
    auto run = [&] (auto logm_c, auto logw_c) -> int
    {
        constexpr int LOGM = decltype (logm_c)::value, LOGW = decltype (logw_c)::value;
        using G = Geo<LOGM, 16>;
        std::vector<float2> tw ((size_t) G::TW_LEN + 1), rtw ((size_t) G::M / 2 + 1);
        fill_stage_twiddles<LOGM, 16> (tw.data());
        fill_real_twiddles (rtw.data(), G::M);
        PConvArgs a { in, in_stride, ir, ir_ch_stride, fdl, fdl_ch_stride, out, out_stride, channels, P, t, scaling, tw.data(), rtw.data() };
        PConvAcc x { acc, acc_stride, S, s_stride };
        emu::g_log_smem = false;
        using PL = PConvLaunch<LOGM>;
        const dim3 grid ((unsigned) ((channels + PL::PER_CTA - 1) / PL::PER_CTA)), block (PL::THREADS);
        if (mode == PCONV_EMIT && S == nullptr)
            emu::launch (pconv_acc_kernel<LOGM, LOGW, PCONV_EMIT, false>, grid, block, (size_t) PL::SMEM_BYTES, a, x);
        else if (mode == PCONV_ADD && S == nullptr)
            emu::launch (pconv_acc_kernel<LOGM, LOGW, PCONV_ADD, false>, grid, block, (size_t) PL::SMEM_BYTES, a, x);
        else if (mode == PCONV_ADD)
            emu::launch (pconv_acc_kernel<LOGM, LOGW, PCONV_ADD, true>, grid, block, (size_t) PL::SMEM_BYTES, a, x);
        else
            return -1;
        return 0;
    };
    using std::integral_constant;
    if (logM == 4 && logW == 2) return run (integral_constant<int, 4> {}, integral_constant<int, 2> {});
    if (logM == 7 && logW == 3) return run (integral_constant<int, 7> {}, integral_constant<int, 3> {});
    if (logM == 8 && logW == 3) return run (integral_constant<int, 8> {}, integral_constant<int, 3> {});
    return -1;
}

// sliced tail multiply-accumulate: pairs [pair0, pair0 + pairs) of S = sum_{p=1}^{P-1} X_(q-p) H_p
void emu_pconv_slice (const float* ir, long long ir_ch_stride, const float* fdl, long long fdl_ch_stride, float* S, long long s_stride, int channels, int P, int N, int logW, int q, int pair0, int pairs)
{
    const PConvSliceArgs a { ir, ir_ch_stride, fdl, fdl_ch_stride, S, s_stride, channels, P, N, logW, q, pair0, pairs };
    const long long items = (long long) channels * pairs;
    emu::g_log_smem = false;
    emu::launch (pconv_slice_kernel, dim3 ((unsigned) ((items + 255) / 256)), dim3 (256), (size_t) 0, a);
}

// the convolver's partition schedule (the library calls the same conv_schedule)
int emu_conv_schedule (int B, long long L, int Bmax, int* block, long long* parts, long long* start, int max_segments)
{
    return conv_schedule (B, L, Bmax, block, parts, start, max_segments);
}
} // extern "C"
