// TEST INFRASTRUCTURE ONLY -- the streaming convolver's IR-swap kernel modes (pconv_kernel.cuh: FROM_FDL, PCONV_EMIT_MIX) run on
// the host through cuda_emu.h, beside the fused modes they must match.  Built into its own library by
// tests/test_emu_convolver_swap.py; not part of the product, never loaded by the package.
#define CHOWDSP_EMU 1
#include "fft_kernels.cuh"
#include "pconv_kernel.cuh"

using namespace cfb;

extern "C"
{
// one launch of pconv_acc_kernel: mode 1 = PCONV_ADD, 2 = PCONV_EMIT, 3 = PCONV_EMIT_MIX; S != nullptr = PARTIAL; from_fdl = X_t
// from delay-line slot t % P.  Only the combinations the library instantiates are accepted.
int emu_pconv_swap (int logM, int logW, int mode, int from_fdl, const float* in, long long in_stride, const float* ir, long long ir_ch_stride,
                    float* fdl, long long fdl_ch_stride, float* out, long long out_stride, float* acc, long long acc_stride, const float* S,
                    long long s_stride, int channels, int P, int t, float scaling, float mix_start, float mix_step)
{
    auto run = [&] (auto logm_c, auto logw_c) -> int
    {
        constexpr int LOGM = decltype (logm_c)::value, LOGW = decltype (logw_c)::value;
        using G = Geo<LOGM, 16>;
        std::vector<float2> tw ((size_t) G::TW_LEN + 1), rtw ((size_t) G::M / 2 + 1);
        fill_stage_twiddles<LOGM, 16> (tw.data());
        fill_real_twiddles (rtw.data(), G::M);
        PConvArgs a { in, in_stride, ir, ir_ch_stride, fdl, fdl_ch_stride, out, out_stride, channels, P, t, scaling, tw.data(), rtw.data() };
        PConvAcc x { acc, acc_stride, S, s_stride, mix_start, mix_step };
        emu::g_log_smem = false;
        using PL = PConvLaunch<LOGM>;
        const dim3 grid ((unsigned) ((channels + PL::PER_CTA - 1) / PL::PER_CTA)), block (PL::THREADS);
        const size_t smem = (size_t) PL::SMEM_BYTES;
        if (! from_fdl && mode == PCONV_EMIT && S == nullptr)
            emu::launch (pconv_acc_kernel<LOGM, LOGW, PCONV_EMIT, false>, grid, block, smem, a, x);
        else if (! from_fdl && mode == PCONV_ADD)
            S == nullptr ? emu::launch (pconv_acc_kernel<LOGM, LOGW, PCONV_ADD, false>, grid, block, smem, a, x)
                         : emu::launch (pconv_acc_kernel<LOGM, LOGW, PCONV_ADD, true>, grid, block, smem, a, x);
        else if (from_fdl && mode == PCONV_ADD)
            S == nullptr ? emu::launch (pconv_acc_kernel<LOGM, LOGW, PCONV_ADD, false, true>, grid, block, smem, a, x)
                         : emu::launch (pconv_acc_kernel<LOGM, LOGW, PCONV_ADD, true, true>, grid, block, smem, a, x);
        else if (from_fdl && mode == PCONV_EMIT_MIX && S == nullptr)
            emu::launch (pconv_acc_kernel<LOGM, LOGW, PCONV_EMIT_MIX, false, true>, grid, block, smem, a, x);
        else
            return -1;
        return 0;
    };
    using std::integral_constant;
    if (logM == 4 && logW == 2) return run (integral_constant<int, 4> {}, integral_constant<int, 2> {});
    if (logM == 7 && logW == 3) return run (integral_constant<int, 7> {}, integral_constant<int, 3> {});
    return -1;
}
} // extern "C"
