// TEST INFRASTRUCTURE ONLY -- runs the CUDA kernel source on the host through cuda_emu.h so that the
// index maps, twiddle tables, layouts and bank-conflict behaviour can be checked without a GPU
// (tests/test_emu_kernels.py, `-m "not gpu"`).  Not part of the product; never loaded by the package.
#define CHOWDSP_EMU 1
#include "fft_kernels.cuh"
#include "elementwise_kernels.cuh"
#include "pconv_kernel.cuh"
#include "pipe_kernels.cuh"
#include "cluster_kernels.cuh"
#include "mixed_kernels.cuh"
#include "mixq_kernels.cuh"
#include "large_plan.h"

using namespace cfb;

namespace
{
int g_emu_radix = 16; // emu_set_radix: 32 selects the 32-points-per-thread geometry where it is instantiated

template <int LOGM, int KIND, int LOGW, int R>
int run_one_r (FftArgs a)
{
    using G = Geo<LOGM, R>;
    using L = Launch<LOGM, R>;
    std::vector<float2> tw ((size_t) G::TW_LEN + 1), rtw ((size_t) G::M / 2 + 1);
    fill_stage_twiddles<LOGM, R> (tw.data());
    fill_real_twiddles (rtw.data(), G::M);
    a.tw = tw.data();
    a.rtw = rtw.data();
    const unsigned grid = (unsigned) ((a.batch + L::PER_CTA - 1) / L::PER_CTA);
    emu::launch (fft_kernel<LOGM, R, KIND, LOGW>, dim3 (grid), dim3 (L::THREADS), (size_t) (LOGW != 0 ? L::SMEM_BYTES_UNORD : L::SMEM_BYTES), a);
    return 0;
}
template <int LOGM, int KIND, int LOGW>
int run_one (FftArgs a)
{
    if constexpr (LOGM == 9 || LOGM == 10 || LOGM == 13 || LOGM == 14)
        if (g_emu_radix == 32)
            return run_one_r<LOGM, KIND, LOGW, 32> (a);
    return g_emu_radix == 16 ? run_one_r<LOGM, KIND, LOGW, 16> (a) : -1;
}

template <int LOGM>
int run_logm (int kind, int logW, const FftArgs& a)
{
    switch (kind * 4 + logW)
    {
        case 0: return run_one<LOGM, C2C_FWD, 0> (a);
        case 2: return run_one<LOGM, C2C_FWD, 2> (a);
        case 4: return run_one<LOGM, C2C_BWD, 0> (a);
        case 6: return run_one<LOGM, C2C_BWD, 2> (a);
        case 8: return run_one<LOGM, R2C, 0> (a);
        case 10: return run_one<LOGM, R2C, 2> (a);
        case 12: return run_one<LOGM, C2R, 0> (a);
        case 14: return run_one<LOGM, C2R, 2> (a);
    }
    if constexpr (LOGM >= 6)
    {
        switch (kind * 4 + logW)
        {
            case 3: return run_one<LOGM, C2C_FWD, 3> (a);
            case 7: return run_one<LOGM, C2C_BWD, 3> (a);
            case 11: return run_one<LOGM, R2C, 3> (a);
            case 15: return run_one<LOGM, C2R, 3> (a);
        }
    }
    return -1;
}
} // namespace

namespace
{
// multi-pass complex transform of 2^n points through the tile kernels (factors forced by the caller so that
// small sizes can exercise the two- and three-pass plans); in/out interleaved complex, natural order
template <int LOGL, int C, int DIR, int R>
void emu_tile_launch_cr (const TilePass& p)
{
    using TL = TileLaunch<LOGL, C, R>;
    const dim3 grid ((unsigned) p.args.ntiles * (unsigned) p.args.batch), block (TL::THREADS);
    if (p.uio == 1)
    {
        if constexpr (DIR > 0)
            emu::launch (tile_fft_kernel<LOGL, C, +1, false, 1, R>, grid, block, (size_t) TL::SMEM_BYTES, p.args);
    }
    else if (p.uio == 2)
    {
        if constexpr (DIR < 0)
            emu::launch (tile_fft_kernel<LOGL, C, -1, true, 2, R>, grid, block, (size_t) TL::SMEM_BYTES, p.args);
    }
    else if (p.load_j_fast)
        emu::launch (tile_fft_kernel<LOGL, C, DIR, true, 0, R>, grid, block, (size_t) TL::SMEM_BYTES, p.args);
    else
        emu::launch (tile_fft_kernel<LOGL, C, DIR, false, 0, R>, grid, block, (size_t) TL::SMEM_BYTES, p.args);
}
// persistent tensor-map TMA tile kernel on (at most) 3 resident CTAs; false = the pass cannot be expressed as tensor maps
template <int LOGL, int C, int DIR>
bool emu_tile_launch_tma (const TilePass& p)
{
    using TT = TileTmaLaunch<LOGL, C, 16>;
    if constexpr (! TT::FITS || LOGL < 8)
        return false;
    else
    {
        TileTmaSide in, out;
        if (! build_tile_tma (p, in, out))
            return false;
        auto to_map = [] (const TileTmaSide& s)
        {
            TensorMap5 m {};
            m.base = reinterpret_cast<const char*> (s.base);
            for (int i = 0; i < 5; ++i)
            {
                m.dim[i] = s.dims[i];
                m.box[i] = s.box[i];
            }
            for (int i = 0; i < 4; ++i)
                m.stride[i] = s.strides[i];
            return m;
        };
        const TensorMap5 im = to_map (in), om = to_map (out);
        const unsigned tiles = (unsigned) p.args.ntiles * (unsigned) p.args.batch, grid = tiles < 3u ? tiles : 3u;
        if (p.load_j_fast)
            emu::launch (tile_tma_kernel<LOGL, C, DIR, true, 16>, dim3 (grid), dim3 (TT::THREADS), (size_t) TT::SMEM_BYTES, im, om, p.args, in.coords, out.coords);
        else
            emu::launch (tile_tma_kernel<LOGL, C, DIR, false, 16>, dim3 (grid), dim3 (TT::THREADS), (size_t) TT::SMEM_BYTES, im, om, p.args, in.coords, out.coords);
        return true;
    }
}
template <int LOGL, int C, int DIR>
void emu_tile_launch_c (const TilePass& p)
{
    if (tile_tma_mode() != 0 && tile_radix32() == 0 && emu_tile_launch_tma<LOGL, C, DIR> (p))
        return;
    if constexpr (LOGL >= 9 && (C == 8 || LOGL == 9))
        if (tile_radix32() != 0)
        {
            emu_tile_launch_cr<LOGL, C, DIR, 32> (p);
            return;
        }
    emu_tile_launch_cr<LOGL, C, DIR, 16> (p);
}
template <int LOGL, int DIR>
void emu_tile_launch (const TilePass& p)
{
    if (p.C == 16)
    {
        if constexpr (LOGL <= 9)
            emu_tile_launch_c<LOGL, 16, DIR> (p);
    }
    else
        emu_tile_launch_c<LOGL, 8, DIR> (p);
}
template <int DIR>
int emu_tile_dispatch (const TilePass& p)
{
    switch (p.logL)
    {
        case 6: emu_tile_launch<6, DIR> (p); return 0;
        case 7: emu_tile_launch<7, DIR> (p); return 0;
        case 8: emu_tile_launch<8, DIR> (p); return 0;
        case 9: emu_tile_launch<9, DIR> (p); return 0;
        case 10: emu_tile_launch<10, DIR> (p); return 0;
    }
    return -1;
}
template <int LOGL>
void fill_tw_for (std::vector<float2>& tw)
{
    if constexpr (LOGL >= 9)
        if (tile_radix32() != 0) // must match emu_tile_launch_c
        {
            tw.assign ((size_t) Geo<LOGL, 32>::TW_LEN + 1, float2 { 0, 0 });
            fill_stage_twiddles<LOGL, 32> (tw.data());
            return;
        }
    tw.assign ((size_t) Geo<LOGL, 16>::TW_LEN + 1, float2 { 0, 0 });
    fill_stage_twiddles<LOGL, 16> (tw.data());
}
} // namespace

extern "C"
{
// logM = log2 of the COMPLEX length run by the CTA (N for C2C, N/2 for real transforms)
int emu_fft (int logM, int kind, int unord, int logW, const float* in, float* out, int batch, int inner, long long in_inner, long long in_outer, long long out_inner, long long out_outer, int log_conflicts, long* stats /* ops, wavefronts, ideal, worst_x100 */)
{
    FftArgs a {};
    a.in = in;
    a.out = out;
    a.in_inner = in_inner;
    a.in_outer = in_outer;
    a.out_inner = out_inner;
    a.out_outer = out_outer;
    a.inner = inner;
    a.batch = batch;
    emu::g_log_smem = log_conflicts != 0;
    emu::g_stats = {};
    int rc = -1;
    switch (logM)
    {
        case 4: rc = run_logm<4> (kind, unord ? logW : 0, a); break;
        case 5: rc = run_logm<5> (kind, unord ? logW : 0, a); break;
        case 6: rc = run_logm<6> (kind, unord ? logW : 0, a); break;
        case 7: rc = run_logm<7> (kind, unord ? logW : 0, a); break;
        case 8: rc = run_logm<8> (kind, unord ? logW : 0, a); break;
        case 9: rc = run_logm<9> (kind, unord ? logW : 0, a); break;
        case 10: rc = run_logm<10> (kind, unord ? logW : 0, a); break;
        case 11: rc = run_logm<11> (kind, unord ? logW : 0, a); break;
        case 12: rc = run_logm<12> (kind, unord ? logW : 0, a); break;
        case 13: rc = run_logm<13> (kind, unord ? logW : 0, a); break;
        case 14: rc = run_logm<14> (kind, unord ? logW : 0, a); break;
        default: break;
    }
    if (stats)
    {
        stats[0] = emu::g_stats.ops;
        stats[1] = emu::g_stats.wavefronts;
        stats[2] = emu::g_stats.ideal;
        stats[3] = emu::g_stats.worst;
    }
    return rc;
}

} // extern "C"
// staged kernel for dense batches of tiny transforms (fft_small_kernel); -1: kind / layout / size not served by it
namespace
{
template <int LOGM, int KIND, int LOGW>
int emu_small_one (FftArgs a)
{
    using SL = SmallLaunch<LOGM, KIND, LOGW>;
    if constexpr (! SL::APPLIES)
        return -1;
    else
    {
        using G = typename SL::G;
        std::vector<float2> tw ((size_t) G::TW_LEN + 1), rtw ((size_t) G::M / 2 + 1);
        fill_stage_twiddles<LOGM, 16> (tw.data());
        fill_real_twiddles (rtw.data(), G::M);
        a.tw = tw.data();
        a.rtw = rtw.data();
        const unsigned grid = (unsigned) ((a.batch + SL::L::PER_CTA - 1) / SL::L::PER_CTA);
        emu::launch (fft_small_kernel<LOGM, KIND, LOGW>, dim3 (grid), dim3 (SL::L::THREADS), (size_t) SL::SMEM_BYTES, a);
        return 0;
    }
}
template <int LOGM>
int emu_small_logm (int kind, int logW, const FftArgs& a)
{
    switch (kind * 4 + logW)
    {
        case 0: return emu_small_one<LOGM, C2C_FWD, 0> (a);
        case 2: return emu_small_one<LOGM, C2C_FWD, 2> (a);
        case 4: return emu_small_one<LOGM, C2C_BWD, 0> (a);
        case 6: return emu_small_one<LOGM, C2C_BWD, 2> (a);
        case 8: return emu_small_one<LOGM, R2C, 0> (a);
        case 10: return emu_small_one<LOGM, R2C, 2> (a);
        case 12: return emu_small_one<LOGM, C2R, 0> (a);
        case 14: return emu_small_one<LOGM, C2R, 2> (a);
    }
    return -1;
}
} // namespace
extern "C"
{
int emu_small (int logM, int kind, int logW, const float* in, float* out, int batch, int log_conflicts, long* stats)
{
    FftArgs a {};
    a.in = in;
    a.out = out;
    a.in_inner = a.out_inner = 2LL << logM;
    a.inner = batch;
    a.batch = batch;
    emu::g_log_smem = log_conflicts != 0;
    emu::g_stats = {};
    int rc = -1;
    switch (logM)
    {
        case 4: rc = emu_small_logm<4> (kind, logW, a); break;
        case 5: rc = emu_small_logm<5> (kind, logW, a); break;
        default: break;
    }
    if (stats)
    {
        stats[0] = emu::g_stats.ops;
        stats[1] = emu::g_stats.wavefronts;
        stats[2] = emu::g_stats.ideal;
        stats[3] = emu::g_stats.worst;
    }
    return rc;
}

// persistent TMA-pipelined transform (pipe_kernels.cuh): `grid` resident CTAs loop over `batch` contiguous transforms
int emu_pipe (int logM, int kind, int unord, const float* in, float* out, int batch, int grid, int log_conflicts, long* stats)
{
    auto run = [&] (auto logm_c, auto logw_c) -> int
    {
        constexpr int LOGM = decltype (logm_c)::value, LOGW = decltype (logw_c)::value;
        using P = PipeGeo<LOGM>;
        using G = typename P::G;
        std::vector<float2> tw ((size_t) G::TW_LEN + 1), rtw ((size_t) G::M / 2 + 1);
        fill_stage_twiddles<LOGM, 32> (tw.data());
        fill_real_twiddles (rtw.data(), G::M);
        FftArgs a {};
        a.in = in; a.out = out;
        a.in_inner = a.out_inner = (kind >= 2 ? 2 : 2) * (long long) G::M;
        a.inner = batch; a.batch = batch;
        a.tw = tw.data(); a.rtw = rtw.data();
        switch (kind)
        {
            case 0: emu::launch (pipe_kernel<LOGM, C2C_FWD, LOGW>, dim3 ((unsigned) grid), dim3 (P::T), (size_t) PipeGeo<LOGM, C2C_FWD, LOGW>::SMEM_BYTES, a); break;
            case 1: emu::launch (pipe_kernel<LOGM, C2C_BWD, LOGW>, dim3 ((unsigned) grid), dim3 (P::T), (size_t) PipeGeo<LOGM, C2C_BWD, LOGW>::SMEM_BYTES, a); break;
            case 2: emu::launch (pipe_kernel<LOGM, R2C, LOGW>, dim3 ((unsigned) grid), dim3 (P::T), (size_t) PipeGeo<LOGM, R2C, LOGW>::SMEM_BYTES, a); break;
            case 3: emu::launch (pipe_kernel<LOGM, C2R, LOGW>, dim3 ((unsigned) grid), dim3 (P::T), (size_t) PipeGeo<LOGM, C2R, LOGW>::SMEM_BYTES, a); break;
            default: return -1;
        }
        return 0;
    };
    emu::g_log_smem = log_conflicts != 0;
    emu::g_stats = {};
    int rc = -1;
    if (logM == 13 && ! unord) rc = run (std::integral_constant<int, 13> {}, std::integral_constant<int, 0> {});
    if (logM == 14 && ! unord) rc = run (std::integral_constant<int, 14> {}, std::integral_constant<int, 0> {});
    if (logM == 13 && unord) rc = run (std::integral_constant<int, 13> {}, std::integral_constant<int, 3> {});
    if (logM == 14 && unord) rc = run (std::integral_constant<int, 14> {}, std::integral_constant<int, 3> {});
    if (stats)
    {
        stats[0] = emu::g_stats.ops;
        stats[1] = emu::g_stats.wavefronts;
        stats[2] = emu::g_stats.ideal;
        stats[3] = emu::g_stats.worst;
    }
    return rc;
}

// the transform kernels with the JUCE adapter's conventions (fft_kernel_juce): kind 1 = C2C_BWD, 2 = R2C, 3 = C2R
int emu_fft_juce (int logM, int radix, int kind, const float* in, float* out, int batch, long long in_stride, long long out_stride)
{
    auto run = [&] (auto logm_c, auto r_c) -> int
    {
        constexpr int LOGM = decltype (logm_c)::value, R = decltype (r_c)::value;
        using G = Geo<LOGM, R>;
        using L = Launch<LOGM, R>;
        std::vector<float2> tw ((size_t) G::TW_LEN + 1), rtw ((size_t) G::M / 2 + 1);
        fill_stage_twiddles<LOGM, R> (tw.data());
        fill_real_twiddles (rtw.data(), G::M);
        FftArgs a {};
        a.in = in; a.out = out; a.in_inner = in_stride; a.out_inner = out_stride; a.inner = a.batch = batch;
        a.tw = tw.data(); a.rtw = rtw.data();
        const unsigned grid = (unsigned) ((batch + L::PER_CTA - 1) / L::PER_CTA);
        emu::g_log_smem = false;
        switch (kind)
        {
            case 1: emu::launch (fft_kernel_juce<LOGM, R, C2C_BWD>, dim3 (grid), dim3 (L::THREADS), (size_t) L::SMEM_BYTES, a); break;
            case 2: emu::launch (fft_kernel_juce<LOGM, R, R2C>, dim3 (grid), dim3 (L::THREADS), (size_t) L::SMEM_BYTES, a); break;
            case 3: emu::launch (fft_kernel_juce<LOGM, R, C2R>, dim3 (grid), dim3 (L::THREADS), (size_t) L::SMEM_BYTES, a); break;
            default: return -1;
        }
        return 0;
    };
    using std::integral_constant;
    if (logM == 4 && radix == 16) return run (integral_constant<int, 4> {}, integral_constant<int, 16> {});
    if (logM == 7 && radix == 16) return run (integral_constant<int, 7> {}, integral_constant<int, 16> {});
    if (logM == 10 && radix == 32) return run (integral_constant<int, 10> {}, integral_constant<int, 32> {});
    if (logM == 11 && radix == 16) return run (integral_constant<int, 11> {}, integral_constant<int, 16> {});
    return -1;
}

// frame-gather R2C (stft_kernel): `outer` channels x `inner` frames, hop = in_inner, optional window
int emu_stft (int logM, int unord, int logW, const float* in, float* out, int outer, int inner, long long in_outer, long long in_inner, long long out_outer, long long out_inner, const float* window, int vec4, int union_gather, int log_conflicts, long* stats)
{
    auto run = [&] (auto logm_c, auto logw_c) -> int
    {
        constexpr int LOGM = decltype (logm_c)::value, LOGW = decltype (logw_c)::value;
        using G = Geo<LOGM, 16>;
        using L = Launch<LOGM, 16>;
        std::vector<float2> tw ((size_t) G::TW_LEN + 1), rtw ((size_t) G::M / 2 + 1);
        fill_stage_twiddles<LOGM, 16> (tw.data());
        fill_real_twiddles (rtw.data(), G::M);
        FftArgs a {};
        a.in = in; a.out = out;
        a.in_inner = in_inner; a.in_outer = in_outer; a.out_inner = out_inner; a.out_outer = out_outer;
        a.inner = inner; a.batch = outer * inner;
        a.tw = tw.data(); a.rtw = rtw.data();
        a.window = window; a.vec4 = vec4;
        a.groups = (inner + L::PER_CTA - 1) / L::PER_CTA;
        a.union_gather = union_gather;
        if (union_gather)
            emu::launch (stft_kernel<LOGM, 16, LOGW, true>, dim3 ((unsigned) (outer * a.groups)), dim3 (L::THREADS), (size_t) (LOGW != 0 ? L::SMEM_BYTES_UNORD : L::SMEM_BYTES), a);
        else
            emu::launch (stft_kernel<LOGM, 16, LOGW, false>, dim3 ((unsigned) (outer * a.groups)), dim3 (L::THREADS), (size_t) (LOGW != 0 ? L::SMEM_BYTES_UNORD : L::SMEM_BYTES), a);
        return 0;
    };
    using std::integral_constant;
    emu::g_log_smem = log_conflicts != 0;
    emu::g_stats = {};
    int rc = -1;
    const int lw = unord ? logW : 0;
#define CFB_EMU_STFT(M, W) if (logM == M && lw == W) rc = run (integral_constant<int, M> {}, integral_constant<int, W> {});
    CFB_EMU_STFT (4, 0) CFB_EMU_STFT (4, 2) CFB_EMU_STFT (6, 0) CFB_EMU_STFT (6, 3) CFB_EMU_STFT (8, 0) CFB_EMU_STFT (8, 3)
    CFB_EMU_STFT (10, 0) CFB_EMU_STFT (10, 3) CFB_EMU_STFT (10, 2) CFB_EMU_STFT (12, 0)
#undef CFB_EMU_STFT
    if (stats)
    {
        stats[0] = emu::g_stats.ops;
        stats[1] = emu::g_stats.wavefronts;
        stats[2] = emu::g_stats.ideal;
        stats[3] = emu::g_stats.worst;
    }
    return rc;
}

// persistent TMA-fed frame gather (stft_pipe_kernel) on `grid` resident CTAs
int emu_stft_pipe (int logM, int radix, int unord, int logW, const float* in, float* out, int outer, int inner, long long in_outer, long long in_inner, long long out_outer, long long out_inner, const float* window, int grid, int log_conflicts, long* stats)
{
    auto run = [&] (auto logm_c, auto r_c, auto logw_c) -> int
    {
        constexpr int LOGM = decltype (logm_c)::value, R = decltype (r_c)::value, LOGW = decltype (logw_c)::value;
        using SP = StftPipeGeo<LOGM, R, LOGW>;
        using G = Geo<LOGM, R>;
        using L = Launch<LOGM, R>;
        std::vector<float2> tw ((size_t) G::TW_LEN + 1), rtw ((size_t) G::M / 2 + 1);
        fill_stage_twiddles<LOGM, R> (tw.data());
        fill_real_twiddles (rtw.data(), G::M);
        FftArgs a {};
        a.in = in; a.out = out;
        a.in_inner = in_inner; a.in_outer = in_outer; a.out_inner = out_inner; a.out_outer = out_outer;
        a.inner = inner; a.batch = outer * inner;
        a.tw = tw.data(); a.rtw = rtw.data();
        a.window = window;
        a.groups = (inner + L::PER_CTA - 1) / L::PER_CTA;
        a.land_bytes = SP::land_bytes (in_inner);
        emu::launch (stft_pipe_kernel<LOGM, R, LOGW>, dim3 ((unsigned) grid), dim3 (L::THREADS), (size_t) SP::smem_bytes (in_inner), a);
        return 0;
    };
    using std::integral_constant;
    emu::g_log_smem = log_conflicts != 0;
    emu::g_stats = {};
    int rc = -1;
    const int lw = unord ? logW : 0;
#define CFB_EMU_SP(M, RR, W) if (logM == M && radix == RR && lw == W) rc = run (integral_constant<int, M> {}, integral_constant<int, RR> {}, integral_constant<int, W> {});
    CFB_EMU_SP (4, 16, 0) CFB_EMU_SP (4, 16, 2) CFB_EMU_SP (6, 16, 0) CFB_EMU_SP (6, 16, 3) CFB_EMU_SP (8, 16, 0) CFB_EMU_SP (8, 16, 3)
    CFB_EMU_SP (10, 16, 0) CFB_EMU_SP (10, 32, 0) CFB_EMU_SP (10, 32, 3) CFB_EMU_SP (12, 16, 0)
#undef CFB_EMU_SP
    if (stats)
    {
        stats[0] = emu::g_stats.ops;
        stats[1] = emu::g_stats.wavefronts;
        stats[2] = emu::g_stats.ideal;
        stats[3] = emu::g_stats.worst;
    }
    return rc;
}

// warp-pipelined transform (wpipe_kernel): `grid` resident CTAs of `warps` warps, kind 0 = C2C_FWD, 2 = R2C
int emu_wpipe (int logM, int radix, int kind, int unord, int logW, const float* in, float* out, int outer, int inner, long long in_outer, long long in_inner, long long out_outer, long long out_inner, const float* window, int grid, int warps, int log_conflicts, long* stats)
{
    auto run = [&] (auto logm_c, auto r_c, auto kind_c, auto logw_c) -> int
    {
        constexpr int LOGM = decltype (logm_c)::value, R = decltype (r_c)::value, KIND = decltype (kind_c)::value, LOGW = decltype (logw_c)::value;
        using WP = WPipeGeo<LOGM, R, LOGW>;
        using G = Geo<LOGM, R>;
        std::vector<float2> tw ((size_t) G::TW_LEN + 1), rtw ((size_t) G::M / 2 + 1);
        fill_stage_twiddles<LOGM, R> (tw.data());
        fill_real_twiddles (rtw.data(), G::M);
        FftArgs a {};
        a.in = in; a.out = out;
        a.in_inner = in_inner; a.in_outer = in_outer; a.out_inner = out_inner; a.out_outer = out_outer;
        a.inner = inner; a.batch = outer * inner;
        a.tw = tw.data(); a.rtw = rtw.data();
        a.window = window;
        if (warps <= 0 || warps > WP::MAX_WARPS)
            return -2;
        emu::launch (wpipe_kernel<LOGM, R, KIND, LOGW>, dim3 ((unsigned) grid), dim3 ((unsigned) warps * 32), (size_t) WP::smem_bytes (warps), a);
        return 0;
    };
    using std::integral_constant;
    emu::g_log_smem = log_conflicts != 0;
    emu::g_stats = {};
    int rc = -1;
    const int lw = unord ? logW : 0;
#define CFB_EMU_WP(M, RR, K, W) if (logM == M && radix == RR && kind == K && lw == W) rc = run (integral_constant<int, M> {}, integral_constant<int, RR> {}, integral_constant<int, K> {}, integral_constant<int, W> {});
    CFB_EMU_WP (10, 32, R2C, 0) CFB_EMU_WP (10, 32, R2C, 3) CFB_EMU_WP (10, 32, R2C, 2) CFB_EMU_WP (10, 32, C2C_FWD, 0) CFB_EMU_WP (10, 32, C2C_FWD, 3) CFB_EMU_WP (10, 32, C2C_FWD, 2)
    CFB_EMU_WP (9, 16, R2C, 0) CFB_EMU_WP (9, 16, R2C, 3) CFB_EMU_WP (9, 16, R2C, 2) CFB_EMU_WP (9, 16, C2C_FWD, 0) CFB_EMU_WP (9, 16, C2C_FWD, 3) CFB_EMU_WP (9, 16, C2C_FWD, 2)
#undef CFB_EMU_WP
    if (stats)
    {
        stats[0] = emu::g_stats.ops;
        stats[1] = emu::g_stats.wavefronts;
        stats[2] = emu::g_stats.ideal;
        stats[3] = emu::g_stats.worst;
    }
    return rc;
}

// warp-pipelined overlap-add synthesis (wistft_kernel): hop = 64 hq floats, `grid` CTAs of `warps` warps, segments of seg_frames
int emu_wistft (int logM, int hq, const float* spec, float* sig, int channels, int frames, long long spec_channel_stride, long long spec_frame_stride, long long channel_stride, const float* window, float scale, int seg_frames, int grid, int warps)
{
    auto run = [&] (auto logm_c, auto r_c, auto hq_c) -> int
    {
        constexpr int LOGM = decltype (logm_c)::value, R = decltype (r_c)::value, HQ = decltype (hq_c)::value;
        using WP = WPipeGeo<LOGM, R, 0>;
        using G = Geo<LOGM, R>;
        std::vector<float2> tw ((size_t) G::TW_LEN + 1), rtw ((size_t) G::M / 2 + 1);
        fill_stage_twiddles<LOGM, R> (tw.data());
        fill_real_twiddles (rtw.data(), G::M);
        FftArgs a {};
        a.in = spec; a.out = sig;
        a.in_inner = spec_frame_stride; a.in_outer = spec_channel_stride; a.out_inner = 64 * HQ; a.out_outer = channel_stride;
        a.inner = frames; a.batch = channels * frames;
        a.tw = tw.data(); a.rtw = rtw.data();
        a.window = window;
        a.scale = scale;
        a.seg_frames = seg_frames;
        a.nseg = (frames + seg_frames - 1) / seg_frames;
        if (warps <= 0 || warps > WIstftGeo<LOGM, R>::MAX_WARPS)
            return -2;
        emu::launch (wistft_kernel<LOGM, R, HQ>, dim3 ((unsigned) grid), dim3 ((unsigned) warps * 32), (size_t) WP::smem_bytes (warps), a);
        return 0;
    };
    using std::integral_constant;
    emu::g_log_smem = false;
    int rc = -1;
#define CFB_EMU_WI(M, RR, H) if (logM == M && hq == H) rc = run (integral_constant<int, M> {}, integral_constant<int, RR> {}, integral_constant<int, H> {});
    CFB_EMU_WI (10, 32, 16) CFB_EMU_WI (10, 32, 8) CFB_EMU_WI (10, 32, 4) CFB_EMU_WI (9, 16, 8) CFB_EMU_WI (9, 16, 4) CFB_EMU_WI (9, 16, 2)
#undef CFB_EMU_WI
    return rc;
}

// overlap-add synthesis (istft_kernel): `channels` x `frames` spectra -> signals, segments of seg_groups CTA groups
// overlap-add synthesis with register accumulators (ristft_kernel); -1: no such instance
int emu_ristft (int logM, int hq, int logW, const float* spec, float* sig, int channels, int frames, long long spec_channel_stride, long long spec_frame_stride, long long channel_stride, const float* window, float scale, int nseg)
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
        a.seg_frames = (frames + nseg - 1) / nseg;
        a.nseg = (frames + a.seg_frames - 1) / a.seg_frames;
        const long long items = (long long) channels * a.nseg;
        emu::g_log_smem = false;
        emu::launch (ristft_kernel<LOGM, HQ, LOGW>, dim3 ((unsigned) ((items + L::PER_CTA - 1) / L::PER_CTA)), dim3 (L::THREADS),
                     (size_t) (LOGW != 0 ? L::SMEM_BYTES_UNORD : L::SMEM_BYTES), a);
        return 0;
    };
    using std::integral_constant;
    int rc = -1;
#define CFB_EMU_RIS(M, H, W) if (logM == M && hq == H && logW == W) rc = run (integral_constant<int, M> {}, integral_constant<int, H> {}, integral_constant<int, W> {});
    CFB_EMU_RIS (6, 4, 3) CFB_EMU_RIS (6, 2, 0) CFB_EMU_RIS (7, 4, 0) CFB_EMU_RIS (8, 8, 2) CFB_EMU_RIS (8, 4, 3)
    CFB_EMU_RIS (9, 4, 0) CFB_EMU_RIS (9, 8, 3) CFB_EMU_RIS (9, 2, 2)
    CFB_EMU_RIS (10, 4, 3) CFB_EMU_RIS (10, 2, 0)
    CFB_EMU_RIS (11, 4, 0) CFB_EMU_RIS (11, 8, 3)
    CFB_EMU_RIS (12, 4, 0)
#undef CFB_EMU_RIS
    return rc;
}

int emu_istft (int logM, int radix, int unord, int logW, const float* spec, float* sig, int channels, int frames, long long spec_channel_stride, long long spec_frame_stride, long long channel_stride, long long hop, const float* window, float scale, int seg_groups)
{
    auto run = [&] (auto logm_c, auto r_c, auto logw_c) -> int
    {
        constexpr int LOGM = decltype (logm_c)::value, R = decltype (r_c)::value, LOGW = decltype (logw_c)::value;
        using G = Geo<LOGM, R>;
        using L = Launch<LOGM, R>;
        std::vector<float2> tw ((size_t) G::TW_LEN + 1), rtw ((size_t) G::M / 2 + 1);
        fill_stage_twiddles<LOGM, R> (tw.data());
        fill_real_twiddles (rtw.data(), G::M);
        FftArgs a {};
        a.in = spec; a.out = sig;
        a.in_inner = spec_frame_stride; a.in_outer = spec_channel_stride; a.out_inner = hop; a.out_outer = channel_stride;
        a.inner = frames; a.batch = channels * frames;
        a.tw = tw.data(); a.rtw = rtw.data();
        a.window = window;
        a.scale = scale;
        a.vec4 = ((hop & 3) == 0 && (channel_stride & 3) == 0 && (reinterpret_cast<uintptr_t> (sig) & 15) == 0) ? 1 : 0;
        const int groups = (frames + L::PER_CTA - 1) / L::PER_CTA;
        a.seg_frames = seg_groups * L::PER_CTA;
        a.nseg = (groups + seg_groups - 1) / seg_groups;
        const int tail_n = 2 * G::M - (int) hop;
        const size_t smem_bytes = (size_t) (LOGW != 0 ? L::SMEM_BYTES_UNORD : L::SMEM_BYTES) + 2 * ((tail_n + 3) & ~3) * 4;
        emu::g_log_smem = false;
        emu::launch (istft_kernel<LOGM, R, LOGW>, dim3 ((unsigned) (channels * a.nseg)), dim3 (L::THREADS), smem_bytes, a);
        return 0;
    };
    using std::integral_constant;
    const int lw = unord ? logW : 0;
    int rc = -1;
#define CFB_EMU_IS(M, RR, W) if (logM == M && radix == RR && lw == W) rc = run (integral_constant<int, M> {}, integral_constant<int, RR> {}, integral_constant<int, W> {});
    CFB_EMU_IS (4, 16, 0) CFB_EMU_IS (4, 16, 2) CFB_EMU_IS (6, 16, 0) CFB_EMU_IS (6, 16, 3) CFB_EMU_IS (8, 16, 0) CFB_EMU_IS (8, 16, 3)
    CFB_EMU_IS (10, 16, 0) CFB_EMU_IS (10, 32, 0) CFB_EMU_IS (10, 32, 3) CFB_EMU_IS (12, 16, 0)
#undef CFB_EMU_IS
    return rc;
}

// generic mixed-radix transform (mixed_kernels.cuh): M complex points per transform, W = 0 (ordered) / 4 / 8
int emu_mixed (int M, int kind, int W, const float* in, float* out, int batch, long long in_stride, long long out_stride, int grid)
{
    MixedArgs a {};
    a.in = in; a.out = out; a.in_stride = in_stride; a.out_stride = out_stride; a.batch = batch;
    a.M = M;
    a.nstages = mixed_factor (M, a.radix);
    if (a.nstages == 0 || M > kMixedMaxM)
        return -1;
    std::vector<float2> w ((size_t) M), r ((size_t) M / 2 + 1);
    fill_mixed_twiddles (w.data(), M);
    fill_mixed_real_twiddles (r.data(), M);
    a.wtab = w.data(); a.rtab = r.data();
    a.kind = kind; a.W = W;
    emu::g_log_smem = false;
    int threads = 0;
    mixed_geometry (M, threads, a.tg);
    emu::launch (mixed_kernel<0>, dim3 ((unsigned) grid), dim3 (threads), (size_t) 16 * M * (threads / a.tg), a);
    return 0;
}

} // extern "C" (the templates below need C++ linkage)
// Q x 2^p mixed-radix transform (mixq_kernels.cuh); -1: no such instance
namespace
{
template <int LOGP, int Q>
int emu_mixq_one (MixQArgs a, int M)
{
    using X = MixQGeo<LOGP, Q>;
    if constexpr (X::M > kMixedMaxM || X::THREADS > 1024)
        return -1;
    else
    {
        std::vector<float2> tw ((size_t) X::G::TW_LEN + 1), w ((size_t) M), r ((size_t) M / 2 + 1);
        fill_stage_twiddles<LOGP, 16> (tw.data());
        fill_mixed_twiddles (w.data(), M);
        fill_mixed_real_twiddles (r.data(), M);
        a.tw = tw.data(); a.wtab = w.data(); a.rtab = r.data();
        emu::g_log_smem = false;
        const bool fast = (a.kind == C2C_FWD || a.kind == C2C_BWD) && a.W == 0;
        emu::launch (fast ? mixq_kernel<LOGP, Q, 0> : mixq_kernel<LOGP, Q, 1>, dim3 ((unsigned) ((a.batch + X::SLOTS - 1) / X::SLOTS)), dim3 (X::THREADS), (size_t) X::SMEM_BYTES, a);
        return 0;
    }
}
template <int LOGP>
int emu_mixq_p (int Q, const MixQArgs& a, int M)
{
    switch (Q)
    {
        case 3: return emu_mixq_one<LOGP, 3> (a, M);
        case 5: return emu_mixq_one<LOGP, 5> (a, M);
        case 9: return emu_mixq_one<LOGP, 9> (a, M);
        case 15: return emu_mixq_one<LOGP, 15> (a, M);
    }
    return -1;
}
} // namespace
extern "C"
{
int emu_mixq (int M, int kind, int W, const float* in, float* out, int batch, long long in_stride, long long out_stride)
{
    int logP = 0, Q = 0;
    if (! mixq_applies (M, logP, Q))
        return -1;
    MixQArgs a {};
    a.in = in; a.out = out; a.in_stride = in_stride; a.out_stride = out_stride; a.batch = batch; a.kind = kind; a.W = W;
    switch (logP)
    {
        case 4: return emu_mixq_p<4> (Q, a, M);
        case 5: return emu_mixq_p<5> (Q, a, M);
        case 6: return emu_mixq_p<6> (Q, a, M);
        case 7: return emu_mixq_p<7> (Q, a, M);
        case 8: return emu_mixq_p<8> (Q, a, M);
        case 9: return emu_mixq_p<9> (Q, a, M);
        case 10: return emu_mixq_p<10> (Q, a, M);
        case 11: return emu_mixq_p<11> (Q, a, M);
        case 12: return emu_mixq_p<12> (Q, a, M);
    }
    return -1;
}

// fused partitioned-convolution step, real size N = 2^(logM+1)
int emu_pconv (int logM, int logW, const float* in, long long in_stride, const float* ir, long long ir_ch_stride, float* fdl, long long fdl_ch_stride, float* out, long long out_stride, int channels, int P, int t, float scaling)
{
    auto run = [&] (auto logm_c, auto logw_c) -> int
    {
        constexpr int LOGM = decltype (logm_c)::value, LOGW = decltype (logw_c)::value;
        using G = Geo<LOGM, 16>;
        std::vector<float2> tw ((size_t) G::TW_LEN + 1), rtw ((size_t) G::M / 2 + 1);
        fill_stage_twiddles<LOGM, 16> (tw.data());
        fill_real_twiddles (rtw.data(), G::M);
        PConvArgs a { in, in_stride, ir, ir_ch_stride, fdl, fdl_ch_stride, out, out_stride, channels, P, t, scaling, tw.data(), rtw.data() };
        emu::g_log_smem = false;
        using PL = PConvLaunch<LOGM>;
        emu::launch (pconv_kernel<LOGM, LOGW>, dim3 ((unsigned) ((channels + PL::PER_CTA - 1) / PL::PER_CTA)), dim3 (PL::THREADS), (size_t) PL::SMEM_BYTES, a);
        return 0;
    };
    using std::integral_constant;
    if (logM == 7 && logW == 3) return run (integral_constant<int, 7> {}, integral_constant<int, 3> {});
    if (logM == 7 && logW == 2) return run (integral_constant<int, 7> {}, integral_constant<int, 2> {});
    if (logM == 4 && logW == 2) return run (integral_constant<int, 4> {}, integral_constant<int, 2> {});
    if (logM == 10 && logW == 3) return run (integral_constant<int, 10> {}, integral_constant<int, 3> {});
    if (logM == 12 && logW == 3) return run (integral_constant<int, 12> {}, integral_constant<int, 3> {});
    return -1;
}

void emu_set_tile_c (int c) { tile_c_override() = c; }
void emu_set_tile_r (int r) { tile_radix32() = r; }
void emu_set_tile_tma (int v) { tile_tma_mode() = v; }
void emu_set_radix (int r) { g_emu_radix = r; }

// batch transforms of 2^n complex points through build_large_schedule: classic whole-array passes (chunk_elems = 0) or the
// L2-chunked schedule (the lanes run one after the other here: this checks the chunk addressing, not the overlap);
// unordered = the W = 2^logW lane layout on the spectrum side (output of forward, input of backward transforms)
int emu_large_c2c (int n, int l1, int l2, int l3, int backward, int batch, int unordered_logW, long long chunk_elems, int lanes, const float* in, float* out, int log_conflicts, long* stats)
{
    LargeFactors f;
    f.l1 = l1; f.l2 = l2; f.l3 = l3;
    if (l1 + l2 + l3 != n)
        return -2;
    const int lobits = big_twiddle_lobits (n);
    std::vector<float2> lo ((size_t) 1 << lobits), hi ((size_t) 1 << (n - lobits));
    fill_big_twiddles (lo.data(), hi.data(), n, lobits);
    const long long N = 1LL << n;
    std::vector<float2> s1 ((size_t) (N * batch));
    const long long ring_lane = ring_elems_needed (n, f, batch, chunk_elems);
    std::vector<float2> ring ((size_t) (ring_lane * lanes) + 1);
    std::vector<float2> tw[3];
    const int logs[3] = { l1, l2, l3 };
    for (int i = 0; i < 3; ++i)
        switch (logs[i])
        {
            case 0: break;
            case 6: fill_tw_for<6> (tw[i]); break;
            case 7: fill_tw_for<7> (tw[i]); break;
            case 8: fill_tw_for<8> (tw[i]); break;
            case 9: fill_tw_for<9> (tw[i]); break;
            case 10: fill_tw_for<10> (tw[i]); break;
            default: return -3;
        }
    emu::g_log_smem = log_conflicts != 0;
    emu::g_stats = {};
    LargeBuffers bufs {};
    bufs.src = reinterpret_cast<const float2*> (in);
    bufs.dst = reinterpret_cast<float2*> (out);
    bufs.src_bs = bufs.dst_bs = N;
    bufs.s1 = s1.data();
    bufs.ring = chunk_elems > 0 ? ring.data() : nullptr;
    bufs.ring_lane_elems = ring_lane;
    std::vector<LargeLaunch> sched;
    build_large_schedule (n, f, batch, bufs, 1u, unordered_logW != 0 && backward, unordered_logW != 0 && ! backward, unordered_logW, chunk_elems, lanes, true, sched);
    for (auto& l : sched)
    {
        l.pass.args.tw = tw[l.pass.which].data();
        l.pass.args.tw_lo = lo.data();
        l.pass.args.tw_hi = hi.data();
        l.pass.args.tw_lobits = lobits;
        const int rc = backward ? emu_tile_dispatch<+1> (l.pass) : emu_tile_dispatch<-1> (l.pass);
        if (rc != 0)
            return rc;
    }
    if (stats)
    {
        stats[0] = emu::g_stats.ops;
        stats[1] = emu::g_stats.wavefronts;
        stats[2] = emu::g_stats.ideal;
        stats[3] = emu::g_stats.worst;
        stats[4] = (long) sched.size();
    }
    return 0;
}

// one local phase of the distributed four-step (large_plan.h: build_dist_phase); forward only
int emu_dist_phase (int n, int l1, int l2, int l3, int phase, int rank, int world, const float* in, float* out)
{
    LargeFactors f;
    f.l1 = l1; f.l2 = l2; f.l3 = l3;
    TilePass p;
    if (! build_dist_phase (n, f, phase, rank, world, p))
        return -2;
    const int lobits = big_twiddle_lobits (n);
    std::vector<float2> lo ((size_t) 1 << lobits), hi ((size_t) 1 << (n - lobits)), tw;
    fill_big_twiddles (lo.data(), hi.data(), n, lobits);
    switch (p.logL)
    {
        case 6: fill_tw_for<6> (tw); break;
        case 7: fill_tw_for<7> (tw); break;
        case 8: fill_tw_for<8> (tw); break;
        case 9: fill_tw_for<9> (tw); break;
        case 10: fill_tw_for<10> (tw); break;
        default: return -3;
    }
    p.args.tw = tw.data();
    p.args.tw_lo = lo.data();
    p.args.tw_hi = hi.data();
    p.args.tw_lobits = lobits;
    p.args.in = reinterpret_cast<const float2*> (in);
    p.args.out = reinterpret_cast<float2*> (out);
    emu::g_log_smem = false;
    return emu_tile_dispatch<-1> (p);
}

// phase 0 with the fused exchange: row block h is stored into outs[h] (exchange layout [world][L1/world][cols])
int emu_dist_phase0_peer (int n, int l1, int l2, int l3, int rank, int world, const float* in, float* const* outs)
{
    LargeFactors f;
    f.l1 = l1; f.l2 = l2; f.l3 = l3;
    TilePass p;
    if (! build_dist_phase (n, f, 0, rank, world, p) || world > 8)
        return -2;
    const int lobits = big_twiddle_lobits (n);
    std::vector<float2> lo ((size_t) 1 << lobits), hi ((size_t) 1 << (n - lobits)), tw;
    fill_big_twiddles (lo.data(), hi.data(), n, lobits);
    switch (p.logL)
    {
        case 6: fill_tw_for<6> (tw); break;
        case 7: fill_tw_for<7> (tw); break;
        case 8: fill_tw_for<8> (tw); break;
        case 9: fill_tw_for<9> (tw); break;
        case 10: fill_tw_for<10> (tw); break;
        default: return -3;
    }
    int wl = 0;
    while ((1 << wl) < world)
        ++wl;
    p.args.tw = tw.data();
    p.args.tw_lo = lo.data();
    p.args.tw_hi = hi.data();
    p.args.tw_lobits = lobits;
    p.args.in = reinterpret_cast<const float2*> (in);
    p.args.out = nullptr;
    p.args.peer_row_log = l1 - wl;
    for (int h = 0; h < world; ++h)
        p.args.peer_out[h] = reinterpret_cast<float2*> (outs[h]);
    emu::g_log_smem = false;
    return emu_tile_dispatch<-1> (p);
}

// phases 1 + 2 of one rank through build_dist_schedule (fft_dist_transform's schedule): recv = this rank's exchange-layout
// buffer; natural = 0: out = transposed-out buffer of this rank; natural = 1: outs[h] = rank h's natural-order block (the
// second all-to-all done by pass C's stores).  chunk_elems = 0: whole-array passes.
int emu_dist_schedule (int n, int l1, int l2, int l3, int rank, int world, int natural, long long chunk_elems, int lanes, const float* recv, float* out, float* const* outs)
{
    LargeFactors f;
    f.l1 = l1; f.l2 = l2; f.l3 = l3;
    const long long S1 = 1LL << (l2 + l3), rows = (1LL << l1) / world;
    const int lobits = big_twiddle_lobits (n);
    std::vector<float2> lo ((size_t) 1 << lobits), hi ((size_t) 1 << (n - lobits));
    fill_big_twiddles (lo.data(), hi.data(), n, lobits);
    std::vector<float2> tw[3];
    const int logs[3] = { l1, l2, l3 };
    for (int i = 1; i < 3; ++i)
        switch (logs[i])
        {
            case 6: fill_tw_for<6> (tw[i]); break;
            case 7: fill_tw_for<7> (tw[i]); break;
            case 8: fill_tw_for<8> (tw[i]); break;
            case 9: fill_tw_for<9> (tw[i]); break;
            case 10: fill_tw_for<10> (tw[i]); break;
            default: return -3;
        }
    const int c_last = tile_c (l3, true);
    long long nrc = chunk_elems / S1;
    nrc -= nrc % c_last;
    if (chunk_elems > 0 && nrc < c_last)
        nrc = c_last;
    const long long ring_lane = chunk_elems > 0 ? (nrc > rows ? rows : nrc) * S1 : 0;
    std::vector<float2> s1 ((size_t) (rows * S1)), ring ((size_t) (ring_lane * lanes) + 1);
    float2* peer_nat[8] = {};
    for (int h = 0; h < world && natural; ++h)
        peer_nat[h] = reinterpret_cast<float2*> (outs[h]);
    std::vector<LargeLaunch> sched;
    if (! build_dist_schedule (n, f, rank, world, reinterpret_cast<const float2*> (recv), natural ? nullptr : reinterpret_cast<float2*> (out), peer_nat, natural != 0,
                               s1.data(), chunk_elems > 0 ? ring.data() : nullptr, ring_lane, chunk_elems, lanes, true, sched))
        return -2;
    emu::g_log_smem = false;
    for (auto& l : sched)
    {
        l.pass.args.tw = tw[l.pass.which].data();
        l.pass.args.tw_lo = lo.data();
        l.pass.args.tw_hi = hi.data();
        l.pass.args.tw_lobits = lobits;
        const int rc = emu_tile_dispatch<-1> (l.pass);
        if (rc != 0)
            return rc;
    }
    return (int) sched.size();
}

// one-pass cluster transform (cluster_kernels.cuh): `nclusters` resident clusters of 2^logG CTAs loop over `batch` contiguous
// transforms of 2^(13 + logG) complex points; unord = 1: 8-lane unordered output (forward only)
int emu_cluster_fft (int logG, int backward, int unord, const float* in, float* out, int batch, int nclusters, int log_conflicts, long* stats)
{
    auto run = [&] (auto logg_c) -> int
    {
        constexpr int LOGG = decltype (logg_c)::value;
        using CG = ClusterGeo<LOGG>;
        constexpr int LOGN = CG::LOGN;
        const long long N = 1LL << LOGN;
        std::vector<float2> tw ((size_t) CG::GL::TW_LEN + 1);
        fill_stage_twiddles<9, 32> (tw.data());
        const int lobits = big_twiddle_lobits (LOGN);
        std::vector<float2> lo ((size_t) 1 << lobits), hi ((size_t) 1 << (LOGN - lobits));
        fill_big_twiddles (lo.data(), hi.data(), LOGN, lobits);
        TensorMap4 tm {};
        tm.base = reinterpret_cast<const char*> (in);
        tm.dim[0] = 32; tm.dim[1] = CG::G; tm.dim[2] = CG::LC; tm.dim[3] = (unsigned long long) batch;
        tm.stride[0] = 128; tm.stride[1] = 128ull * CG::G; tm.stride[2] = (unsigned long long) N * 8;
        tm.box[0] = 32; tm.box[1] = 1; tm.box[2] = CG::TMA_ROWS; tm.box[3] = 1;
        ClusterArgs a {};
        a.out = out;
        a.out_stride = 2 * N;
        a.batch = batch;
        a.logW = unord ? 3 : 0;
        a.tw = tw.data();
        a.tw_lo = lo.data();
        a.tw_hi = hi.data();
        a.tw_lobits = lobits;
        a.l2_prefetch = 1;
        TensorMap4 om {};
        om.base = reinterpret_cast<const char*> (out);
        om.dim[0] = 1024; om.dim[1] = 16 * CG::G; om.dim[2] = (unsigned long long) batch;
        om.stride[0] = 4096; om.stride[1] = (unsigned long long) N * 8;
        om.box[0] = 2 * CG::RUN; om.box[1] = 16 * CG::G; om.box[2] = 1;
        const dim3 grid ((unsigned) (nclusters * CG::G)), block (CG::THREADS);
        if (backward)
            emu::launch_cluster (cluster_fft_kernel<LOGG, +1, 0>, grid, CG::G, block, (size_t) CG::SMEM_BYTES, tm, om, a);
        else if (unord)
            emu::launch_cluster (cluster_fft_kernel<LOGG, -1, 3>, grid, CG::G, block, (size_t) CG::SMEM_BYTES, tm, om, a);
        else
            emu::launch_cluster (cluster_fft_kernel<LOGG, -1, 0>, grid, CG::G, block, (size_t) CG::SMEM_BYTES, tm, om, a);
        return 0;
    };
    emu::g_log_smem = log_conflicts != 0;
    emu::g_stats = {};
    int rc = -1;
    if (logG == 1) rc = run (std::integral_constant<int, 1> {});
    if (logG == 2) rc = run (std::integral_constant<int, 2> {});
    if (logG == 3) rc = run (std::integral_constant<int, 3> {});
    if (stats)
    {
        stats[0] = emu::g_stats.ops;
        stats[1] = emu::g_stats.wavefronts;
        stats[2] = emu::g_stats.ideal;
        stats[3] = emu::g_stats.worst;
    }
    return rc;
}

int emu_convolve (const float* a, const float* b, float* ab, long long a_stride, long long b_stride, long long ab_stride, int nfloats, int batch, int logW, int is_real, float scaling)
{
    ConvArgs p { a, b, ab, a_stride, b_stride, ab_stride, nfloats, batch, logW, is_real, scaling };
    emu::launch (convolve_kernel, dim3 (2), dim3 (64), 0, p);
    return 0;
}

int emu_accumulate (const float* a, const float* b, float* ab, long long n)
{
    emu::launch (accumulate_kernel, dim3 (2), dim3 (64), 0, a, b, ab, n / 4);
    return 0;
}
}
