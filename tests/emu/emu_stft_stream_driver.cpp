// TEST INFRASTRUCTURE ONLY -- streaming overlap-add synthesis (ristft_body with CARRY, fft_kernels.cuh) runs on the host through
// cuda_emu.h, beside the offline ristft_kernel it must match bit for bit.  Built into its own library by
// tests/test_emu_stft_stream.py; not part of the product, never loaded by the package.
#define CHOWDSP_EMU 1
#include "fft_kernels.cuh"

using namespace cfb;

extern "C"
{
// one launch of overlap-add synthesis over `frames` spectra per channel: carry == nullptr = ristft_kernel in nseg segments (the
// offline kernel, whole channels), else ristft_carry_kernel with its accumulators loaded from and stored to carry ((N - hop) / 2
// float2 per channel).  -1: no such instance.
int emu_ristft_stream (int logM, int hq, int logW, const float* spec, float* sig, int channels, int frames, long long spec_channel_stride, long long spec_frame_stride,
                       long long channel_stride, const float* window, float scale, int nseg, float* carry)
{
    auto run = [&] (auto logm_c, auto hq_c, auto logw_c) -> int
    {
        constexpr int LOGM = decltype (logm_c)::value, HQ = decltype (hq_c)::value, LOGW = decltype (logw_c)::value;
        using G = Geo<LOGM, 16>;
        using L = Launch<LOGM, 16>;
        std::vector<float2> tw ((size_t) G::TW_LEN + 1), rtw ((size_t) G::M / 2 + 1);
        fill_stage_twiddles<LOGM, 16> (tw.data());
        fill_real_twiddles (rtw.data(), G::M);
        FftArgs a {};
        a.in = spec; a.out = sig;
        a.in_inner = spec_frame_stride; a.in_outer = spec_channel_stride; a.out_inner = 2 * G::T * HQ; a.out_outer = channel_stride;
        a.inner = frames; a.batch = channels * frames;
        a.tw = tw.data(); a.rtw = rtw.data();
        a.window = window;
        a.scale = scale;
        a.seg_frames = carry != nullptr ? frames : (frames + nseg - 1) / nseg;
        a.nseg = (frames + a.seg_frames - 1) / a.seg_frames;
        const long long items = (long long) channels * a.nseg;
        const dim3 grid ((unsigned) ((items + L::PER_CTA - 1) / L::PER_CTA)), block (L::THREADS);
        const size_t smem = (size_t) (LOGW != 0 ? L::SMEM_BYTES_UNORD : L::SMEM_BYTES);
        emu::g_log_smem = false;
        if (carry != nullptr)
            emu::launch (ristft_carry_kernel<LOGM, HQ, LOGW>, grid, block, smem, a, reinterpret_cast<float2*> (carry));
        else
            emu::launch (ristft_kernel<LOGM, HQ, LOGW>, grid, block, smem, a);
        return 0;
    };
    using std::integral_constant;
    int rc = -1;
#define CFB_EMU_RS(M, H, W) if (logM == M && hq == H && logW == W) rc = run (integral_constant<int, M> {}, integral_constant<int, H> {}, integral_constant<int, W> {});
#define CFB_EMU_RS_M(M) CFB_EMU_RS (M, 2, 0) CFB_EMU_RS (M, 4, 0) CFB_EMU_RS (M, 8, 0) CFB_EMU_RS (M, 2, 3) CFB_EMU_RS (M, 4, 3) CFB_EMU_RS (M, 8, 3)
    CFB_EMU_RS_M (6) CFB_EMU_RS_M (9) CFB_EMU_RS_M (11)
    CFB_EMU_RS (9, 4, 2)
#undef CFB_EMU_RS_M
#undef CFB_EMU_RS
    return rc;
}
} // extern "C"
