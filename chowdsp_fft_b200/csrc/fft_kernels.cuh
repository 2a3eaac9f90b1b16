// Single-kernel shared-memory Stockham FFT for sm_100a: batched power-of-2 fp32 C2C / R2C / C2R,
// ordered and "unordered" (the reference's SIMD-blocked layout), M = 2^4 .. 2^14 complex points per CTA.
//
// This replaces, on the GPU, the reference's whole per-transform pipeline
//   uninterleave -> cfftf1_ps/rfftf1_ps passes -> pffft_cplx_finalize / pffft_real_finalize -> pffft_zreorder
//   (/root/reference/simd/chowdsp_fft_impl_avx.cpp:1848-1935 and the passes at :206-490, :719-1013,
//    :1016-1351, :1354-1689, :1693-1839)
// with ONE launch that reads each input element from HBM once and writes each output element once.
// It is not a translation of the FFTPACK passes: each thread keeps R (=16) complex points in registers,
// runs radix-16 butterflies, and exchanges data between stages through padded shared memory
// (Stockham autosort, so no bit reversal pass); the real transforms are an N/2-point complex FFT with
// the split/merge step fused in, and the output permutation (natural order or the reference's
// unordered layout, SURVEY.md §8a-L) is applied in the epilogue's addressing.
//
// The same source compiles for the host with -DCHOWDSP_EMU (tests/emu): test infrastructure that
// checks index maps / bank conflicts without a GPU.  The product only ever builds the nvcc path.
#pragma once

#ifdef CHOWDSP_EMU
#include "cuda_emu.h"
#define FFT_HD inline
#define FFT_CX constexpr
#define FFT_DYN_SMEM(type, name) type* name = reinterpret_cast<type*> (emu::ctx.smem)
#else
#include <cuda_runtime.h>
#include <type_traits>
#define FFT_HD __device__ __forceinline__
#define FFT_CX __host__ __device__ constexpr
#define FFT_DYN_SMEM(type, name)                   \
    extern __shared__ __align__ (16) char name##_raw[]; \
    type* name = reinterpret_cast<type*> (name##_raw)
#endif

namespace cfb
{
// ---------------------------------------------------------------------------------------------
// transform kinds / kernel arguments
// ---------------------------------------------------------------------------------------------
enum Kind : int
{
    C2C_FWD = 0, // interleaved complex in  -> spectrum out
    C2C_BWD = 1, // spectrum in             -> interleaved complex out
    R2C = 2,     // N real in               -> half spectrum out (N floats)
    C2R = 3      // half spectrum in        -> N real out
};

struct FftArgs
{
    const float* in;
    float* out;
    // transform x = outer * inner + i   reads  in + outer * in_outer + i * in_inner   (floats);
    // plain batches use inner = batch, outer stride 0.  The two-level form is the STFT frame gather.
    long long in_inner, in_outer, out_inner, out_outer;
    int inner;
    int batch;           // total transforms
    const float2* tw;    // stage twiddles, see twiddle_table_len()
    const float2* rtw;   // real split twiddles exp(-2 pi i k / N) / 2, k < N/4 (R2C / C2R only)
    // frame-gather (STFT) kernels only: optional analysis / synthesis window of N floats (nullptr = rectangular),
    // CTA groups per outer index (= ceil (inner / transforms per CTA)), 128-bit global accesses allowed
    const float* window;
    int groups;
    int vec4;
    int union_gather;    // stage the union of a CTA's frames through shared memory (see stft_kernel)
    // L2 prefetch distance in CTAs (0 = off): a CTA asks L2 for the input of CTA blockIdx.x + pf_ahead, about one
    // wave of resident CTAs ahead, so that the loads of a later CTA on this SM find their lines in L2
    int pf_ahead;
    // persistent frame-gather kernel (stft_pipe_kernel): bytes of its landing buffer, ((PER_CTA - 1) hop + N) * 4
    int land_bytes;
    // overlap-add synthesis (istft_kernel): frames per segment (a multiple of the CTA's transforms), segments per
    // channel, output scale
    int seg_frames, nseg;
    float scale;
};

// ---------------------------------------------------------------------------------------------
// geometry
// ---------------------------------------------------------------------------------------------
FFT_CX int ilog2 (int v) { return v <= 1 ? 0 : 1 + ilog2 (v >> 1); }
FFT_CX int ipow (int b, int e) { return e == 0 ? 1 : b * ipow (b, e - 1); }

template <int LOGM_, int R_>
struct Geo
{
    static constexpr int LOGM = LOGM_;
    static constexpr int M = 1 << LOGM_;                 // complex points per transform
    static constexpr int R = R_;                         // complex points held per thread
    static constexpr int LOGR = ilog2 (R_);
    static constexpr int T = M / R;                      // threads per transform
    static constexpr int S = (LOGM + LOGR - 1) / LOGR;   // stages
    static constexpr int RLAST = 1 << (LOGM - (S - 1) * LOGR);
    static constexpr int SMEM_F2 = M + (M >> LOGR);      // padded float2 slots per transform (one pad slot per R)
    static constexpr int SMEM_F2_UNORD = M + (M >> 3);   // staging image of the unordered layout (W=4 pad is the larger one)
    static_assert (M >= R, "transform smaller than the per-thread radix");
    static FFT_CX int radix (int s) { return s == S - 1 ? RLAST : R; }
    static FFT_CX int ns (int s) { return ipow (R, s); } // product of the radices before stage s
    // Stage twiddle tables (stage 0 has none), all holding forward twiddles exp(-2 pi i k q / (Ns r)):
    //   full-radix stage (r = R): rows q in {1, 2, 3} and {4, 8, .., R-4} x Ns entries (6 rows for R = 16, 10
    //                    for R = 32); every other power is one product of two rows (w^q = w^(q%4) w^(q-q%4)),
    //                    computed in registers
    //   last stage r < R: (r-1) rows q = 1..r-1 x T entries (k = j only); the R/r butterflies of a thread
    //                    differ by the constant factors W_R^(u q), applied with immediates
    static_assert (R_ == 16 || R_ == 32, "the twiddle scheme below assumes 16 or 32 points per thread");
    static constexpr int FULL_ROWS = 3 + (R_ / 4 - 1);
    static FFT_CX int tw_rows (int s) { return radix (s) == R ? FULL_ROWS * ns (s) : (radix (s) - 1) * T; }
    // one padding slot per R float2: stride-2^a accesses (2^a <= R) and unit-stride accesses are both conflict
    // free, pad (a + b) = pad (a) + pad (b) whenever R | b, so every offset used below folds into an immediate
    static FFT_CX int pad (int i) { return i + (i >> LOGR); }
    static FFT_CX int tw_off (int s) { return s <= 1 ? 0 : tw_off (s - 1) + tw_rows (s - 1); }
    static constexpr int TW_LEN = S == 1 ? 0 : tw_off (S - 1) + tw_rows (S - 1);
};


// ---------------------------------------------------------------------------------------------
// memory helpers (shared-memory ones are instrumented in the emulator)
// ---------------------------------------------------------------------------------------------
// streaming global loads: read-only path, no L1 allocation (the inputs are touched once; the twiddle
// tables are what should stay in L1)
FFT_HD float2 ldg_stream (const float2* p)
{
#ifdef CHOWDSP_EMU
    return *p;
#else
    float2 r;
    asm volatile ("ld.global.nc.L1::no_allocate.v2.f32 {%0, %1}, [%2];" : "=f"(r.x), "=f"(r.y) : "l"(p));
    return r;
#endif
}
FFT_HD float4 ldg_stream (const float4* p)
{
#ifdef CHOWDSP_EMU
    return *p;
#else
    float4 r;
    asm volatile ("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
#endif
}

// input loads of fft_core: streaming (no L1 allocation) when the T threads of a transform cover a whole 128-byte line with every load
// instruction (T >= 16); with fewer threads per transform every line is touched by 2 .. 16 different instructions of the warp, so there
// the first touch allocates the line in L1 and the others hit instead of going to L2 again (one or two threads per transform even
// split 32-byte sectors: ncu l1tex sectors 2-4x the algorithmic figure with no_allocate)
template <int T>
FFT_HD float2 ldg_in (const float2* p)
{
#if defined(CHOWDSP_EMU) || defined(CFB_NO_CACHED_SMALL_LOADS)
    return ldg_stream (p);
#else
#ifndef CFB_CACHED_LOADS_MAX_T
#define CFB_CACHED_LOADS_MAX_T 8 // burst-mode A/B on B200 (profiles/r02_retune.txt): up to 8 threads per transform +1..13 %, nothing beyond
#endif
    if constexpr (T <= CFB_CACHED_LOADS_MAX_T)
        return __ldg (p);
    else
        return ldg_stream (p);
#endif
}

template <int T>
FFT_HD float4 ldg_in (const float4* p)
{
#if defined(CHOWDSP_EMU) || defined(CFB_NO_CACHED_SMALL_LOADS)
    return ldg_stream (p);
#else
    if constexpr (T <= CFB_CACHED_LOADS_MAX_T)
        return __ldg (p);
    else
        return ldg_stream (p);
#endif
}

// ask L2 for the 128-byte lines of one transform's input (M complex = M/16 lines, R/16 per thread)
template <class G>
FFT_HD void prefetch_transform_l2 (const float* p, int j)
{
#ifndef CHOWDSP_EMU
#pragma unroll
    for (int i = 0; i < (G::R >= 16 ? G::R / 16 : 1); ++i)
        asm volatile ("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char*> (p) + (size_t) (j + i * G::T) * 128));
#else
    (void) p;
    (void) j;
#endif
}

// orders this thread's earlier generic-proxy shared-memory accesses before later async-proxy (bulk copy) accesses
FFT_HD void fence_proxy_async()
{
#ifndef CHOWDSP_EMU
    asm volatile ("fence.proxy.async.shared::cta;" ::: "memory");
#endif
}

FFT_HD void prefetch_l2 (const void* p)
{
#ifndef CHOWDSP_EMU
    asm volatile ("prefetch.global.L2 [%0];" ::"l"(p));
#else
    (void) p;
#endif
}

FFT_HD float2 lds2 (const float2* p)
{
#ifdef CHOWDSP_EMU
    if (emu::ctx.log)
        emu::ctx.log->push_back ({ (uint32_t) ((const char*) p - emu::ctx.smem), 8, 0 });
#endif
    return *p;
}
FFT_HD void sts2 (float2* p, float2 v)
{
#ifdef CHOWDSP_EMU
    if (emu::ctx.log)
        emu::ctx.log->push_back ({ (uint32_t) ((const char*) p - emu::ctx.smem), 8, 1 });
#endif
    *p = v;
}
FFT_HD void smem_skip() // keeps the per-warp op sequences aligned when a lane is predicated off
{
#ifdef CHOWDSP_EMU
    if (emu::ctx.log)
        emu::ctx.log->push_back ({ 0, 0, 0 });
#endif
}

// value of `v` held by lane `src` of this thread's group of `width` lanes (width = power of two <= 32; every lane of
// the warp must call it)
FFT_HD float2 shfl2 (float2 v, int src, int width)
{
#ifdef CHOWDSP_EMU
    return make_float2 (emu::shfl (v.x, src, width), emu::shfl (v.y, src, width));
#else
    return make_float2 (__shfl_sync (0xffffffffu, v.x, src, width), __shfl_sync (0xffffffffu, v.y, src, width));
#endif
}
FFT_HD float shfl1 (float v, int src, int width)
{
#ifdef CHOWDSP_EMU
    return emu::shfl (v, src, width);
#else
    return __shfl_sync (0xffffffffu, v, src, width);
#endif
}
#ifndef CFB_UNORD_DIRECT
#define CFB_UNORD_DIRECT 1 // A/B switch (tools/ only): 0 = unordered complex spectra always go through the shared-memory staging image
#endif
#ifndef CFB_UNORD_REAL_DIRECT
#define CFB_UNORD_REAL_DIRECT 0
#endif
#ifndef CFB_REAL_TW_DERIVE
#define CFB_REAL_TW_DERIVE 2 // real split / merge twiddles of fft_core: 0 = one table load per bin, 1 = derived in registers, 2 = measured policy (RTW_DERIVE)
#endif
#ifndef CFB_SHFL_MIRROR
#define CFB_SHFL_MIRROR 1 // A/B switch (tools/ only): 0 = the real split / merge step of fft_kernel exchanges through shared memory
#endif

// ---------------------------------------------------------------------------------------------
// complex arithmetic.  DIR = -1 forward (e^{-i..}), +1 backward.
// ---------------------------------------------------------------------------------------------
// Blackwell packed fp32x2 math (SASS FADD2 / FMUL2 / FFMA2): one instruction per COMPLEX add, two per
// complex multiply.  The operand modifiers of those instructions (half swap, per-half negate, scalar
// broadcast) absorb the (y, x) / (-y, x) shuffles written below, so multiplying by +-i is free.
#ifdef CHOWDSP_EMU
FFT_HD float2 f2_add (float2 a, float2 b) { return make_float2 (a.x + b.x, a.y + b.y); }
FFT_HD float2 f2_sub (float2 a, float2 b) { return make_float2 (a.x - b.x, a.y - b.y); }
FFT_HD float2 f2_mul (float2 a, float2 b) { return make_float2 (a.x * b.x, a.y * b.y); }
FFT_HD float2 f2_fma (float2 a, float2 b, float2 c) { return make_float2 (std::fmaf (a.x, b.x, c.x), std::fmaf (a.y, b.y, c.y)); }
#else
FFT_HD unsigned long long f2_bits (float2 v) { return *reinterpret_cast<unsigned long long*> (&v); }
FFT_HD float2 f2_from (unsigned long long b) { return *reinterpret_cast<float2*> (&b); }
FFT_HD float2 f2_add (float2 a, float2 b)
{
    unsigned long long r;
    asm ("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(f2_bits (a)), "l"(f2_bits (b)));
    return f2_from (r);
}
FFT_HD float2 f2_sub (float2 a, float2 b)
{
    unsigned long long r;
    asm ("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(f2_bits (a)), "l"(f2_bits (b)));
    return f2_from (r);
}
FFT_HD float2 f2_mul (float2 a, float2 b)
{
    unsigned long long r;
    asm ("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(f2_bits (a)), "l"(f2_bits (b)));
    return f2_from (r);
}
FFT_HD float2 f2_fma (float2 a, float2 b, float2 c)
{
    unsigned long long r;
    asm ("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(f2_bits (a)), "l"(f2_bits (b)), "l"(f2_bits (c)));
    return f2_from (r);
}
#endif

FFT_HD float2 cadd (float2 a, float2 b) { return f2_add (a, b); }
FFT_HD float2 csub (float2 a, float2 b) { return f2_sub (a, b); }
// a * w (DIR < 0) or a * conj(w) (DIR > 0); tables always hold the forward twiddle
template <int DIR>
FFT_HD float2 cmul_dir (float2 a, float2 w)
{
    const float2 t = f2_mul (a, make_float2 (w.x, w.x));
    if (DIR < 0)
        return f2_fma (make_float2 (a.y, a.x), make_float2 (-w.y, w.y), t); // (ax wx - ay wy, ay wx + ax wy)
    return f2_fma (make_float2 (a.y, a.x), make_float2 (w.y, -w.y), t);     // (ax wx + ay wy, ay wx - ax wy)
}
// a * (-i) forward, a * (+i) backward
template <int DIR>
FFT_HD float2 mul_mi (float2 a)
{
    return DIR < 0 ? make_float2 (a.y, -a.x) : make_float2 (-a.y, a.x);
}
// cos (2 pi n / 32), sin (2 pi n / 32) as compile-time constants
FFT_CX float cos32 (int n)
{
    n &= 31;
    if (n > 16)
        n = 32 - n;
    const bool neg = n > 8;
    if (neg)
        n = 16 - n;
    const float c = n == 0 ? 1.f : n == 1 ? 0.980785280403230449f : n == 2 ? 0.923879532511286756f : n == 3 ? 0.831469612302545237f
                  : n == 4 ? 0.707106781186547524f : n == 5 ? 0.555570233019602225f : n == 6 ? 0.382683432365089772f
                  : n == 7 ? 0.195090322016128268f : 0.f;
    return neg ? -c : c;
}
FFT_CX float sin32 (int n) { return cos32 (n + 24); }

// a * exp(DIR * 2 pi i * NUM / 32) with compile-time constants
template <int DIR, int NUM>
FFT_HD float2 mul_w32 (float2 a)
{
    constexpr int n = NUM & 31;
    if (n == 0)
        return a;
    if (n == 8)
        return mul_mi<DIR> (a);
    if (n == 16)
        return make_float2 (-a.x, -a.y);
    if (n == 24)
        return mul_mi<-DIR> (a);
    return cmul_dir<DIR> (a, make_float2 (cos32 (n), -sin32 (n))); // forward twiddle c - i s
}
template <int DIR, int NUM>
FFT_HD float2 mul_w16 (float2 a) { return mul_w32<DIR, 2 * NUM> (a); }

// a * W32^(DIR * num): num is a loop constant after unrolling, so the switch folds away
template <int DIR>
FFT_HD float2 mul_w32_rt (float2 a, int num)
{
    switch (num & 31)
    {
#define CFB_W32_CASE(n) case n: return mul_w32<DIR, n> (a);
        CFB_W32_CASE (0) CFB_W32_CASE (1) CFB_W32_CASE (2) CFB_W32_CASE (3) CFB_W32_CASE (4) CFB_W32_CASE (5) CFB_W32_CASE (6) CFB_W32_CASE (7)
        CFB_W32_CASE (8) CFB_W32_CASE (9) CFB_W32_CASE (10) CFB_W32_CASE (11) CFB_W32_CASE (12) CFB_W32_CASE (13) CFB_W32_CASE (14) CFB_W32_CASE (15)
        CFB_W32_CASE (16) CFB_W32_CASE (17) CFB_W32_CASE (18) CFB_W32_CASE (19) CFB_W32_CASE (20) CFB_W32_CASE (21) CFB_W32_CASE (22) CFB_W32_CASE (23)
        CFB_W32_CASE (24) CFB_W32_CASE (25) CFB_W32_CASE (26) CFB_W32_CASE (27) CFB_W32_CASE (28) CFB_W32_CASE (29) CFB_W32_CASE (30)
#undef CFB_W32_CASE
        default: return mul_w32<DIR, 31> (a);
    }
}

// cos / sin (pi n / 32), n = 0..32, as compile-time constants (forward twiddles W_64^n = c - i s)
FFT_CX float cos64 (int n)
{
    const bool neg = n > 16;
    if (neg)
        n = 32 - n;
    const float c = n == 0 ? 1.f : n == 1 ? 0.995184726672196886f : n == 2 ? 0.980785280403230449f : n == 3 ? 0.956940335732208865f
                  : n == 4 ? 0.923879532511286756f : n == 5 ? 0.881921264348355030f : n == 6 ? 0.831469612302545237f
                  : n == 7 ? 0.773010453362736961f : n == 8 ? 0.707106781186547524f : n == 9 ? 0.634393284163645498f
                  : n == 10 ? 0.555570233019602225f : n == 11 ? 0.471396736825997649f : n == 12 ? 0.382683432365089772f
                  : n == 13 ? 0.290284677254462368f : n == 14 ? 0.195090322016128268f : n == 15 ? 0.098017140329560602f : 0.f;
    return neg ? -c : c;
}
FFT_CX float sin64 (int n) { return cos64 (n <= 16 ? 16 - n : n - 16); } // n in [0, 32]

// real split / merge twiddle w_k / 2 of bin k = j + m T (T = M / R).  DERIVE = false: one table load per bin (the
// faster choice wherever the table stays in L1: measured -5 % with DERIVE on B200, the FMA pipe is the scarcer unit,
// profiles/r01_real_tw_ab.txt).  DERIVE = true: w_k = w_j W_(2R)^m from the thread's own w_j, a compile-time
// constant after unrolling -- for kernels whose shared-memory carve-out leaves no L1 for a 64 KB table.
template <int R, bool DERIVE>
FFT_HD float2 real_tw (float2 wj, const float2* __restrict__ rt_mT, int m)
{
    if (m == 0)
        return wj;
    if constexpr (! DERIVE)
        return __ldg (rt_mT);
    else if constexpr (R == 16)
        return mul_w32_rt<-1> (wj, m);
    else
        return cmul_dir<-1> (wj, make_float2 (cos64 (m), -sin64 (m)));
}

// ---------------------------------------------------------------------------------------------
// register butterflies: in place, natural-order output, elements v[0], v[ST], v[2 ST], ...
// ---------------------------------------------------------------------------------------------
template <int DIR>
FFT_HD void bfly4 (float2& a0, float2& a1, float2& a2, float2& a3)
{
    const float2 t0 = cadd (a0, a2), t1 = csub (a0, a2), t2 = cadd (a1, a3), t3 = mul_mi<DIR> (csub (a1, a3));
    a0 = cadd (t0, t2);
    a1 = cadd (t1, t3);
    a2 = csub (t0, t2);
    a3 = csub (t1, t3);
}

template <int RADIX, int DIR, int ST>
struct RegFft;

template <int DIR, int ST>
struct RegFft<1, DIR, ST>
{
    static FFT_HD void run (float2*) {}
};
template <int DIR, int ST>
struct RegFft<2, DIR, ST>
{
    static FFT_HD void run (float2* v)
    {
        const float2 a = v[0], b = v[ST];
        v[0] = cadd (a, b);
        v[ST] = csub (a, b);
    }
};
template <int DIR, int ST>
struct RegFft<4, DIR, ST>
{
    static FFT_HD void run (float2* v) { bfly4<DIR> (v[0], v[ST], v[2 * ST], v[3 * ST]); }
};
template <int DIR, int ST>
struct RegFft<8, DIR, ST>
{
    static FFT_HD void run (float2* v)
    {
        float2 e0 = v[0], e1 = v[2 * ST], e2 = v[4 * ST], e3 = v[6 * ST];
        float2 o0 = v[ST], o1 = v[3 * ST], o2 = v[5 * ST], o3 = v[7 * ST];
        bfly4<DIR> (e0, e1, e2, e3);
        bfly4<DIR> (o0, o1, o2, o3);
        o1 = mul_w16<DIR, 2> (o1);
        o2 = mul_mi<DIR> (o2);
        o3 = mul_w16<DIR, 6> (o3);
        v[0] = cadd (e0, o0);      v[4 * ST] = csub (e0, o0);
        v[ST] = cadd (e1, o1);     v[5 * ST] = csub (e1, o1);
        v[2 * ST] = cadd (e2, o2); v[6 * ST] = csub (e2, o2);
        v[3 * ST] = cadd (e3, o3); v[7 * ST] = csub (e3, o3);
    }
};
template <int DIR, int ST>
struct RegFft<16, DIR, ST>
{
    // 16 = 4 x 4:  X[k1 + 4 k2] = sum_n2 W16^(n2 k1) W4^(n2 k2) [ sum_n1 a[4 n1 + n2] W4^(n1 k1) ]
    static FFT_HD void run (float2* v)
    {
        float2 b[4][4]; // b[n2][k1]
#pragma unroll
        for (int n2 = 0; n2 < 4; ++n2)
        {
            b[n2][0] = v[(n2) *ST];
            b[n2][1] = v[(n2 + 4) * ST];
            b[n2][2] = v[(n2 + 8) * ST];
            b[n2][3] = v[(n2 + 12) * ST];
            bfly4<DIR> (b[n2][0], b[n2][1], b[n2][2], b[n2][3]);
        }
        b[1][1] = mul_w16<DIR, 1> (b[1][1]);
        b[1][2] = mul_w16<DIR, 2> (b[1][2]);
        b[1][3] = mul_w16<DIR, 3> (b[1][3]);
        b[2][1] = mul_w16<DIR, 2> (b[2][1]);
        b[2][2] = mul_w16<DIR, 4> (b[2][2]);
        b[2][3] = mul_w16<DIR, 6> (b[2][3]);
        b[3][1] = mul_w16<DIR, 3> (b[3][1]);
        b[3][2] = mul_w16<DIR, 6> (b[3][2]);
        b[3][3] = mul_w16<DIR, 9> (b[3][3]);
#pragma unroll
        for (int k1 = 0; k1 < 4; ++k1)
        {
            bfly4<DIR> (b[0][k1], b[1][k1], b[2][k1], b[3][k1]);
            v[(k1) *ST] = b[0][k1];
            v[(k1 + 4) * ST] = b[1][k1];
            v[(k1 + 8) * ST] = b[2][k1];
            v[(k1 + 12) * ST] = b[3][k1];
        }
    }
};

template <int DIR, int ST>
struct RegFft<32, DIR, ST>
{
    // 32 = 2 x 16:  X[k] = E[k] + W32^k O[k],  X[k + 16] = E[k] - W32^k O[k]
    static FFT_HD void run (float2* v)
    {
        float2 e[16], o[16];
#pragma unroll
        for (int k = 0; k < 16; ++k)
        {
            e[k] = v[(2 * k) * ST];
            o[k] = v[(2 * k + 1) * ST];
        }
        RegFft<16, DIR, 1>::run (e);
        RegFft<16, DIR, 1>::run (o);
#pragma unroll
        for (int k = 0; k < 16; ++k)
        {
            const float2 t = mul_w32_rt<DIR> (o[k], k);
            v[k * ST] = cadd (e[k], t);
            v[(k + 16) * ST] = csub (e[k], t);
        }
    }
};

// ---------------------------------------------------------------------------------------------
// position of a bin inside the reference's unordered layouts (SURVEY.md §8a-L; pffft_zreorder,
// /root/reference/simd/chowdsp_fft_impl_avx.cpp:1780-1839).  Returns the float offset of the real
// part; the imaginary part sits W floats later.
// ---------------------------------------------------------------------------------------------
template <int LOGN> // complex transform of N = 2^LOGN bins
FFT_HD int unordered_pos_complex (int bin, int logW)
{
    const int logL = LOGN - logW;                   // bins per lane row
    const int r = bin >> logL, rem = bin & ((1 << logL) - 1);
    const int b = rem >> logW, lane = rem & ((1 << logW) - 1);
    return ((((b << logW) + r) * 2) << logW) + lane;
}
template <int LOGM> // real transform of 2M samples: bins 0..M-1 (bin 0 carries DC.re and Nyquist.re)
FFT_HD int unordered_pos_real (int bin, int logW)
{
    const int logQ = LOGM - logW, Q = 1 << logQ;
    const int r = bin >> logQ, mr = bin & (Q - 1);
    const int m = (r & 1) ? ((Q - mr) & (Q - 1)) : mr; // odd rows are stored reversed
    const int b = m >> logW, lane = m & ((1 << logW) - 1);
    return ((((b << logW) + r) * 2) << logW) + lane;
}

// Twiddles W^(j q), q = 1 .. r-1, of a short last stage with 32 points per thread: rows q = 1, 2, 3 and 4, 8, .. come
// from load (q), every other power is one product w^(q mod 4) w^(q - q mod 4), as in the full-radix stages.
// pipe_kernel keeps only the loaded rows in shared memory; fft_kernel forms the same products, so a transform gives
// the same bits in either kernel.
template <int r, class Load>
FFT_HD void last_stage_tw (float2 (&w)[r], const Load& load)
{
#pragma unroll
    for (int q = 1; q < r; ++q)
        if (q < 4 || (q & 3) == 0)
            w[q] = load (q);
#pragma unroll
    for (int q = 5; q < r; ++q)
        if ((q & 3) != 0)
            w[q] = cmul_dir<-1> (w[q & 3], w[q & ~3]);
}

// ---------------------------------------------------------------------------------------------
// one Stockham stage on the thread's R registers.  On entry v[m] = x_s[j + m T] (x_s = stage input in
// natural order); on exit of the last stage v[m] = X[j + m T].
// ---------------------------------------------------------------------------------------------
template <class G, int DIR, int STAGE>
FFT_HD void stage_compute (float2 (&v)[G::R], int j, const float2* __restrict__ tw)
{
    constexpr int r = G::radix (STAGE), Ns = G::ns (STAGE), SUB = G::R / r;
    if constexpr (STAGE > 0 && r == G::R && G::R == 16)
    {
        const float2* __restrict__ t = tw + G::tw_off (STAGE) + (j & (Ns - 1));
        const float2 w1 = __ldg (t), w2 = __ldg (t + Ns), w3 = __ldg (t + 2 * Ns);
        const float2 w4 = __ldg (t + 3 * Ns), w8 = __ldg (t + 4 * Ns), w12 = __ldg (t + 5 * Ns);
        v[1] = cmul_dir<DIR> (v[1], w1);
        v[2] = cmul_dir<DIR> (v[2], w2);
        v[3] = cmul_dir<DIR> (v[3], w3);
        v[4] = cmul_dir<DIR> (v[4], w4);
        v[5] = cmul_dir<DIR> (v[5], cmul_dir<-1> (w1, w4));
        v[6] = cmul_dir<DIR> (v[6], cmul_dir<-1> (w2, w4));
        v[7] = cmul_dir<DIR> (v[7], cmul_dir<-1> (w3, w4));
        v[8] = cmul_dir<DIR> (v[8], w8);
        v[9] = cmul_dir<DIR> (v[9], cmul_dir<-1> (w1, w8));
        v[10] = cmul_dir<DIR> (v[10], cmul_dir<-1> (w2, w8));
        v[11] = cmul_dir<DIR> (v[11], cmul_dir<-1> (w3, w8));
        v[12] = cmul_dir<DIR> (v[12], w12);
        v[13] = cmul_dir<DIR> (v[13], cmul_dir<-1> (w1, w12));
        v[14] = cmul_dir<DIR> (v[14], cmul_dir<-1> (w2, w12));
        v[15] = cmul_dir<DIR> (v[15], cmul_dir<-1> (w3, w12));
    }
    else if constexpr (STAGE > 0 && r == G::R)
    {
        // R = 32: rows w^1, w^2, w^3 and w^4, w^8, .., w^28
        const float2* __restrict__ t = tw + G::tw_off (STAGE) + (j & (Ns - 1));
        const float2 w1 = __ldg (t), w2 = __ldg (t + Ns), w3 = __ldg (t + 2 * Ns);
        v[1] = cmul_dir<DIR> (v[1], w1);
        v[2] = cmul_dir<DIR> (v[2], w2);
        v[3] = cmul_dir<DIR> (v[3], w3);
#pragma unroll
        for (int a4 = 1; a4 < G::R / 4; ++a4)
        {
            const float2 wa = __ldg (t + (2 + a4) * Ns);
            v[4 * a4] = cmul_dir<DIR> (v[4 * a4], wa);
            v[4 * a4 + 1] = cmul_dir<DIR> (v[4 * a4 + 1], cmul_dir<-1> (w1, wa));
            v[4 * a4 + 2] = cmul_dir<DIR> (v[4 * a4 + 2], cmul_dir<-1> (w2, wa));
            v[4 * a4 + 3] = cmul_dir<DIR> (v[4 * a4 + 3], cmul_dir<-1> (w3, wa));
        }
    }
    else if constexpr (STAGE > 0 && G::R == 32)
    {
        // last stage, radix r < R, 32 points per thread: the twiddles of pipe_kernel (last_stage_tw), so that the two
        // kernels give the same bits at the sizes both serve
        const float2* __restrict__ t = tw + G::tw_off (STAGE) + j;
        float2 w[r];
        last_stage_tw<r> (w, [&] (int q) { return __ldg (t + (q - 1) * G::T); });
#pragma unroll
        for (int q = 1; q < r; ++q)
        {
#pragma unroll
            for (int u = 0; u < SUB; ++u)
            {
                const float2 x = cmul_dir<DIR> (v[u + q * SUB], w[q]);
                v[u + q * SUB] = mul_w32_rt<DIR> (x, u * q);
            }
        }
    }
    else if constexpr (STAGE > 0)
    {
        // last stage, radix r < R: butterfly u of this thread has k = j + u T, and
        // W^(k q) = W^(j q) W_R^(u q)  because T = M / R
        const float2* __restrict__ t = tw + G::tw_off (STAGE) + j;
#pragma unroll
        for (int q = 1; q < r; ++q)
        {
            const float2 wq = __ldg (t + (q - 1) * G::T);
#pragma unroll
            for (int u = 0; u < SUB; ++u)
            {
                const float2 x = cmul_dir<DIR> (v[u + q * SUB], wq);
                v[u + q * SUB] = mul_w32_rt<DIR> (x, u * q * (32 / G::R));
            }
        }
    }
#pragma unroll
    for (int u = 0; u < SUB; ++u)
        RegFft<r, DIR, SUB>::run (&v[u]);
}

// Shared-memory addressing.  pad() is additive whenever one operand is a multiple of 16, so every
// access below is written as (one per-thread base computed once) + (a compile-time padded offset):
// the offset folds into the LDS/STS immediate and costs no integer instructions.
template <class G, int STAGE>
FFT_HD void stage_scatter (const float2 (&v)[G::R], int j, float2* s)
{
    constexpr int r = G::radix (STAGE), Ns = G::ns (STAGE), SUB = G::R / r;
#pragma unroll
    for (int u = 0; u < SUB; ++u)
    {
        const int jv = j + u * G::T;
        const int k = jv & (Ns - 1);
        const int base = (jv - k) * r + k;
        if constexpr (Ns % G::R == 0)
        {
            float2* sb = s + G::pad (base);
#pragma unroll
            for (int q = 0; q < r; ++q)
                sts2 (sb + G::pad (q * Ns), v[u + q * SUB]);
        }
        else if constexpr (Ns == 1 && r == G::R)
        {
            float2* sb = s + (G::R + 1) * jv; // pad (R jv + q) = (R + 1) jv + q
#pragma unroll
            for (int q = 0; q < r; ++q)
                sts2 (sb + q, v[u + q * SUB]);
        }
        else
        {
#pragma unroll
            for (int q = 0; q < r; ++q)
                sts2 (s + G::pad (base + q * Ns), v[u + q * SUB]);
        }
    }
}

// pointer to natural-order element (j + m T) of the exchange buffer, m in [M0, M1)
template <class G, int M0, int M1>
FFT_HD void gather_natural (float2 (&v)[G::R], int j, const float2* s)
{
    if constexpr (G::T % G::R == 0)
    {
        const float2* sb = s + G::pad (j);
#pragma unroll
        for (int m = M0; m < M1; ++m)
            v[m] = lds2 (sb + G::pad (m * G::T));
    }
    else
    {
#pragma unroll
        for (int m = M0; m < M1; ++m)
            v[m] = lds2 (s + G::pad (j + m * G::T));
    }
}
template <class G, int M0, int M1>
FFT_HD void scatter_natural (const float2 (&v)[G::R], int j, float2* s)
{
    if constexpr (G::T % G::R == 0)
    {
        float2* sb = s + G::pad (j);
#pragma unroll
        for (int m = M0; m < M1; ++m)
            sts2 (sb + G::pad (m * G::T), v[m]);
    }
    else
    {
#pragma unroll
        for (int m = M0; m < M1; ++m)
            sts2 (s + G::pad (j + m * G::T), v[m]);
    }
}
// natural-order slot of the mirror element M - (j + m T), m < R/2 (the caller handles j == 0 && m == 0)
template <class G>
FFT_HD int mirror_slot (int j, int m)
{
    if constexpr (G::T % G::R == 0)
        return G::pad (G::T - j) + G::pad (G::M - m * G::T - G::T); // (M - mT - T) + (T - j), first term % R == 0
    else
        return G::pad (G::M - j - m * G::T);
}

// barrier among the T threads of ONE transform whose shared-memory region is private to it (PRIV): a warp-level
// barrier when the transform fits in a warp, a named barrier (one id per transform of the CTA) for 64 or 128
// threads, the CTA barrier otherwise.  The transforms of a CTA then stop marching in lock step through their load /
// exchange / math phases (ncu on the STFT config: 16 resident warps per SM, barrier + phase-aligned MIO and
// math-pipe stalls; +5..13 % on B200, profiles/r01_transform_barriers.txt).  PRIV = false is the CTA-wide barrier.
template <int T, bool PRIV>
FFT_HD void tsync()
{
    constexpr int MODE = ! PRIV ? 0 : T <= 32 ? 1 : T < 256 ? 2 : 0;
#ifdef CHOWDSP_EMU
    if (MODE == 1)
        emu::syncgroup (32);
    else if (MODE == 2)
        emu::syncgroup (T);
    else
        __syncthreads();
#elif defined(CFB_NO_WARP_SYNC) // A/B switch (tools/ only)
    __syncthreads();
#else
    if (MODE == 1)
        __syncwarp();
    else if (MODE == 2)
        asm volatile ("bar.sync %0, %1;" ::"r"(1 + (int) threadIdx.x / T), "n"(T) : "memory"); // ids 1 .. 256 / T <= 4
    else
        __syncthreads();
#endif
}

struct NoHook
{
    FFT_HD void operator() () const {}
};
// WS: the transform's barriers may be warp-level (see tsync); CTA_FIRST: ... except the first one, which also
// orders the other transforms' reads of a CTA-wide input image (IN_UNION) before this transform's exchange writes
template <class G, int DIR, int STAGE, bool WS = false, bool CTA_FIRST = true>
struct Stages
{
    // from_smem: v was gathered from shared memory just before (a barrier is needed before overwriting it).
    // `input_consumed` runs once, right after the first barrier: every thread of the CTA has then taken its
    // stage-0 input out of shared memory (the persistent kernels start the next input copy there).
    // `last_gathered` (when not NoHook) runs after a barrier that follows the gather of the LAST exchange: from then on
    // the transform does not touch `s` any more unless its epilogue stages an unordered / real-split image there.
    template <class Hook = NoHook, class Hook2 = NoHook>
    static FFT_HD void run (float2 (&v)[G::R], int j, float2* s, const float2* __restrict__ tw, bool from_smem, const Hook& input_consumed = Hook(),
                            const Hook2& last_gathered = Hook2())
    {
        stage_compute<G, DIR, STAGE> (v, j, tw);
        if constexpr (STAGE < G::S - 1)
        {
            if (STAGE > 0 || from_smem)
                tsync<G::T, WS && ! (STAGE == 0 && CTA_FIRST)>(); // every thread has finished reading the previous exchange
            if constexpr (STAGE == 0)
                input_consumed();
            stage_scatter<G, STAGE> (v, j, s);
            tsync<G::T, WS>();
            gather_natural<G, 0, G::R> (v, j, s);
            if constexpr (STAGE == G::S - 2 && ! std::is_same<Hook2, NoHook>::value)
            {
                fence_proxy_async(); // this thread's generic-proxy accesses to `s` are ordered before the async-proxy (TMA) writes the hook starts
                tsync<G::T, WS>();
                last_gathered();
            }
            Stages<G, DIR, STAGE + 1, WS, CTA_FIRST>::run (v, j, s, tw, true, NoHook(), last_gathered);
        }
    }
};

// ---------------------------------------------------------------------------------------------
// unordered I/O goes through a shared-memory staging image of the spectrum IN THE UNORDERED LAYOUT, so
// that global memory only ever sees linear 128-bit accesses; the permutation is paid on-chip.
// Staging pad: one W-float gap per 2 W^2 floats keeps both the scattered 4-byte accesses (runs of W
// lanes at stride 2 W^2) and the linear 16-byte accesses conflict free.
// ---------------------------------------------------------------------------------------------
FFT_HD int upad (int p, int logW) { return p + ((p >> (2 * logW + 1)) << logW); }

FFT_HD float lds1 (const float* p)
{
#ifdef CHOWDSP_EMU
    if (emu::ctx.log)
        emu::ctx.log->push_back ({ (uint32_t) ((const char*) p - emu::ctx.smem), 4, 0 });
#endif
    return *p;
}
FFT_HD void sts1 (float* p, float v)
{
#ifdef CHOWDSP_EMU
    if (emu::ctx.log)
        emu::ctx.log->push_back ({ (uint32_t) ((const char*) p - emu::ctx.smem), 4, 1 });
#endif
    *p = v;
}
FFT_HD float4 lds4 (const float* p)
{
#ifdef CHOWDSP_EMU
    if (emu::ctx.log)
        emu::ctx.log->push_back ({ (uint32_t) ((const char*) p - emu::ctx.smem), 16, 0 });
#endif
    return *reinterpret_cast<const float4*> (p);
}
FFT_HD void sts4 (float* p, float4 v)
{
#ifdef CHOWDSP_EMU
    if (emu::ctx.log)
        emu::ctx.log->push_back ({ (uint32_t) ((const char*) p - emu::ctx.smem), 16, 1 });
#endif
    *reinterpret_cast<float4*> (p) = v;
}

// Padded staging position (float index) of the bins a thread touches, as base(j) + constexpr(m).
//   complex layout: bin j + m T            -> cplx (m)
//   real layout:    bin k = j + m T, m<R/2 -> real_lo (m);   bin M - k -> real_hi (m)
// Derivation: with L = M / W bins per lane row and L / T = R / W =: LT rows-per-... ratio, bin j + m T sits
// in row r = m / LT at in-row index j + (m % LT) T; a row-local index i maps to block b = i / W, lane
// i % W, padded position b (2 W^2 + W) + r 2 W + lane.  Odd rows of the real layout are reversed
// (i -> (Q - i) mod Q), which turns j into -j; the wrap (i == 0) only ever hits thread j == 0 and is
// patched with a select.  Falls back to the generic index computation when T < W.
template <class G, int LOGW, bool PADDED = true> // PADDED = false: float offsets in the unpadded (global-memory) layout
struct UPos
{
    static constexpr int W = 1 << LOGW, PW = 2 * W * W + (PADDED ? W : 0), T = G::T, M = G::M, R = G::R;
    static constexpr int Q = M / W;                       // bins per lane row
    static constexpr int LOGQ = G::LOGM - LOGW;
    static constexpr bool FAST = (T >= W) && (R >= W);
    static constexpr int LT = FAST ? R / W : 1;           // T-sized chunks per lane row
    int j, ub_pos, ub_neg;
    FFT_HD explicit UPos (int j_) : j (j_)
    {
        ub_pos = (j_ >> LOGW) * PW + (j_ & (W - 1));
        ub_neg = ((-j_) >> LOGW) * PW + ((-j_) & (W - 1));
    }
    static FFT_HD int generic_complex (int bin) { return PADDED ? upad (unordered_pos_complex<G::LOGM> (bin, LOGW), LOGW) : unordered_pos_complex<G::LOGM> (bin, LOGW); }
    static FFT_HD int generic_real (int bin) { return PADDED ? upad (unordered_pos_real<G::LOGM> (bin, LOGW), LOGW) : unordered_pos_real<G::LOGM> (bin, LOGW); }

    FFT_HD int cplx (int m) const
    {
        if constexpr (! FAST)
            return generic_complex (j + m * T);
        else
            return ub_pos + (m % LT) * (T / W) * PW + (m / LT) * 2 * W;
    }
    FFT_HD int real_lo (int m) const
    {
        if constexpr (! FAST)
            return generic_real (j + m * T);
        else
        {
            const int r = m / LT, mp = m % LT;
            if ((r & 1) == 0)
                return ub_pos + mp * (T / W) * PW + r * 2 * W;
            const int fast = ub_neg + ((Q - mp * T) / W) * PW + r * 2 * W;
            return (mp == 0 && j == 0) ? r * 2 * W : fast;
        }
    }
    FFT_HD int real_hi (int m) const // bin M - (j + m T); not valid for (j == 0 && m == 0)
    {
        if constexpr (! FAST)
            return generic_real (M - j - m * T);
        else
        {
            const int c = M - m * T;
            const int rr = (c - T) >> LOGQ, e = (c - T) & (Q - 1);
            const int fast = (rr & 1) == 0 ? ub_neg + ((T + e) / W) * PW + rr * 2 * W
                                           : ub_pos + ((Q - e - T) / W) * PW + rr * 2 * W;
            return (c % Q == 0 && j == 0) ? (c >> LOGQ) * 2 * W : fast;
        }
    }
};
template <int LOGW>
FFT_CX int W_HALF_ROW() { return (1 << LOGW) * (1 << LOGW); } // padded staging position of real bin M/2 (row W/2, index 0)
FFT_HD float2 staged_load (const float* sf, int upos, int W) { return make_float2 (lds1 (sf + upos), lds1 (sf + upos + W)); }
FFT_HD void staged_store (float* sf, int upos, int W, float2 v)
{
    sts1 (sf + upos, v.x);
    sts1 (sf + upos + W, v.y);
}
// linear 128-bit copies between global memory and the staging image (2M floats = T * R/2 float4)
template <class G>
FFT_HD void staging_fill (float* sf, const float* __restrict__ in, int j, int logW, bool active)
{
#pragma unroll
    for (int i = 0; i < G::R / 2; ++i)
    {
        const int q = j + i * G::T;
        const float4 val = ldg_in<2 * G::T> (reinterpret_cast<const float4*> (in) + q); // 16 bytes per thread: whole lines from 8 threads on
        sts4 (sf + upad (4 * q, logW), val);
    }
}
template <class G>
FFT_HD void staging_drain (const float* sf, float* __restrict__ out, int j, int logW, bool active)
{
#pragma unroll
    for (int i = 0; i < G::R / 2; ++i)
    {
        const int q = j + i * G::T;
        const float4 val = lds4 (sf + upad (4 * q, logW));
        if (active)
            reinterpret_cast<float4*> (out)[q] = val;
    }
}

// ---------------------------------------------------------------------------------------------
// One transform on the calling thread group (T threads, j = thread index inside the transform).
//   IN_STAGED  (unordered inputs only): the staging image is already in `s` and synchronised
//   OUT_STAGED (unordered outputs only): leave the staging image in `s` (synchronised), do not drain it
//   HALF_OUT   (C2R only): store only the second half of the output samples (overlap-save discard)
//   IN_UNION   (R2C / C2C_FWD, and C2R from an ordered spectrum with mode 2): the stage-0 input is read from the shared-memory image `su` (natural order,
//              unpadded, float2 units; it may alias `s`) and multiplied by the window `win` when non-null.
//              1 = the image is shared by the transforms of the CTA (the first barrier is CTA-wide), 2 = it is
//              private to this transform (wpipe_kernel's per-warp landing buffer: transform-level barriers only)
//   input_consumed (IN_UNION with more than one stage): hook run after the barrier that follows the stage-0 reads
//   last_gathered (more than one stage): hook run after a barrier that follows the gather of the last exchange -- `s` is
//              free from then on for ordered outputs (the warp-pipelined kernels start the next input copy INTO it)
//   OUT_REGS   (C2R / C2C_BWD): do not store; hand the result registers (element j + m T in vout[m]) to the caller
//   FMT = 1    (ordered layouts): the conventions of the reference's JUCE adapter (chowdsp_fft_juce/chowdsp_fft_juce.cpp:
//              32-86) instead of pffft's -- real spectra as N/2 + 1 interleaved complex bins (Nyquist at float 2M, the
//              imaginary parts of DC and Nyquist zero) rather than Nyquist packed into float 1, and inverse transforms
//              (C2R, C2C_BWD) scaled by 1/N
template <int LOGM, int R, int KIND, int LOGW, bool IN_STAGED, bool OUT_STAGED, bool HALF_OUT, int IN_UNION = 0, class Hook = NoHook, bool OUT_REGS = false, int FMT = 0, class Hook2 = NoHook>
FFT_HD void fft_core (const float* __restrict__ in, float* __restrict__ out, bool active, int j, float2* s, const float2* __restrict__ tw_, const float2* __restrict__ rtw_,
                      const float2* su = nullptr, const float2* __restrict__ win = nullptr, const Hook& input_consumed = Hook(), float2* vout = nullptr,
                      const Hook2& last_gathered = Hook2())
{
    using G = Geo<LOGM, R>;
    constexpr int DIR = (KIND == C2C_FWD || KIND == R2C) ? -1 : +1;
    constexpr bool UNORD = LOGW != 0; // 0 = ordered; 2 / 3 = the reference's 4- / 8-lane unordered layout
    constexpr int M = G::M, T = G::T;
    // transforms that own their shared-memory region synchronise among their own threads only (tsync)
    constexpr bool WS = ! IN_STAGED && ! OUT_STAGED;
    // Unordered COMPLEX spectra without the staging image: neighbouring threads (bins j, j+1) swap one float by shuffle, so
    // that the even thread holds (re_j, re_j+1) and the odd one (im_j, im_j+1) -- each a contiguous, 8-byte aligned pair
    // of the unordered layout.  A warp's 64-bit access then covers whole 64-byte [W re | W im] groups: the same
    // instruction count as the ordered path, no shared-memory round trip, no barriers.
    using UPD = UPos<G, UNORD ? LOGW : 2>;
    constexpr bool UDIRECT = CFB_UNORD_DIRECT != 0 && UNORD && UPD::FAST && (KIND == C2C_FWD || KIND == C2C_BWD);
    constexpr int UW = UPD::W, ULT = UPD::LT;
    const int u_odd = j & 1;
    const int u_base = (((j & ~1) >> (UNORD ? LOGW : 2)) * 2 * UW * UW) + ((j & ~1) & (UW - 1)) + (u_odd ? UW : 0); // float offset of this thread's pair
    constexpr int SW = T < 32 ? T : 32; // shuffle width: transforms never straddle a warp
    // Unordered REAL spectra without the staging image (A/B switch CFB_UNORD_REAL_DIRECT): 4-byte accesses straight to the
    // unordered positions; a warp's access still covers whole 32-byte sectors (runs of W lanes)
    constexpr bool RDIRECT = CFB_UNORD_REAL_DIRECT != 0 && UNORD && ((KIND == R2C && ! OUT_STAGED) || (KIND == C2R && ! IN_STAGED));
    const UPos<G, UNORD ? LOGW : 2, false> upg (j);
    // real split / merge: transforms owned by (part of) one warp exchange the mirror half of the spectrum by shuffle
    // (measured, profiles/r01_shfl_mirror.txt: +3..14 % for 16 points per thread and in the warp-pipelined kernels; with
    // 32 points per thread in fft_kernel the 32 extra shuffles + selects cost 2..5 %, so that geometry keeps shared memory)
    constexpr bool SHFL_MIRROR = T <= 32 && (KIND == R2C || KIND == C2R) && ((CFB_SHFL_MIRROR != 0 && R == 16) || IN_UNION == 2);
    // Real split / merge twiddles: derived in registers (w_k = w_j W_2R^m, one table load per thread) or one table load per bin.
    // Burst-mode A/B on B200 (profiles/r02_retune.txt; the round-1 table in profiles/r01_real_tw_ab.txt was taken under the power
    // cap, where the variant with more FMA work loses): the table loads double the global-load sectors of the real kernels
    // (l1tex 77..87 % busy), deriving wins +2..12 % for ordered spectra at every size and for unordered ones up to 2^11 complex
    // points, and loses 1.5 % for unordered 2^12 and 6 % in the warp-pipelined kernel (landing-buffer input), which keep the table.
    // Not below 2^11 complex points (gains of 0..3 % there): those sizes also run in the warp-pipelined kernels, and the host- and
    // device-pointer paths of the STFT entry points, which may pick different kernels, promise bit-identical results.
    // The sizes pipe_kernel also serves (32 points per thread at 2^13 / 2^14) derive them in every layout, as pipe_kernel does: a
    // batch gives the same bits whichever of the two kernels its geometry selects.
    constexpr bool RTW_DERIVE = CFB_REAL_TW_DERIVE == 1
                                || (CFB_REAL_TW_DERIVE == 2 && IN_UNION == 0 && LOGM >= 11 && (! UNORD || LOGM <= 11 || (R == 32 && LOGM >= 13)));
    float* sf = reinterpret_cast<float*> (s); // the same buffer seen as the unordered staging image
    constexpr int logW = LOGW;
    struct { const float2* tw; const float2* rtw; } a { tw_, rtw_ };

    float2 v[R];
    bool smem_was_read = false; // a barrier is needed before the exchange buffer is overwritten
    constexpr int WL = UNORD ? (1 << LOGW) : 1;
    const UPos<G, UNORD ? LOGW : 2> up (j);

    // ---- prologue: v[m] = stage-0 input element j + m T -------------------------------------------
    if constexpr (KIND == C2C_FWD || KIND == R2C || (KIND == C2C_BWD && ! UNORD))
    {
        // interleaved complex (natural order), or real samples read as (x[2n], x[2n+1]) pairs
        if constexpr (IN_UNION != 0)
        {
            const float2* sj = su + j;
#pragma unroll
            for (int m = 0; m < R; ++m)
                v[m] = lds2 (sj + m * T);
            if (win != nullptr)
            {
                const float2* __restrict__ wj = win + j;
#pragma unroll
                for (int m = 0; m < R; ++m)
                    v[m] = f2_mul (v[m], __ldg (wj + m * T));
            }
            smem_was_read = true;
        }
        else
        {
            const float2* __restrict__ in2 = reinterpret_cast<const float2*> (in) + j;
#pragma unroll
            for (int m = 0; m < R; ++m)
                v[m] = ldg_in<T> (in2 + m * T);
            if (win != nullptr) // constant-folded away in the plain batched kernel
            {
                const float2* __restrict__ wj = win + j;
#pragma unroll
                for (int m = 0; m < R; ++m)
                    v[m] = f2_mul (v[m], __ldg (wj + m * T));
            }
        }
    }
    else if constexpr (KIND == C2C_BWD && UDIRECT && ! IN_STAGED)
    {
        const float* __restrict__ ib = in + u_base;
#pragma unroll
        for (int m = 0; m < R; ++m)
        {
            const float2 ld = ldg_in<T> (reinterpret_cast<const float2*> (ib + (m % ULT) * (T / UW) * 2 * UW * UW + (m / ULT) * 2 * UW));
            const float recv = shfl1 (u_odd ? ld.x : ld.y, (j ^ 1) & (SW - 1), SW);
            v[m] = u_odd ? make_float2 (recv, ld.y) : make_float2 (ld.x, recv);
        }
    }
    else if constexpr (KIND == C2C_BWD)
    {
        if constexpr (! IN_STAGED)
        {
            staging_fill<G> (sf, in, j, logW, active);
            tsync<T, WS>();
        }
#pragma unroll
        for (int m = 0; m < R; ++m)
            v[m] = staged_load (sf, up.cplx (m), WL);
        smem_was_read = true;
    }
    else // C2R: merge step  Z'[k] = (X[k] + X*[M-k]) + i conj(w_k) (X[k] - X*[M-k]),  w_k = e^{-2 pi i k / 2M}
    {
        // This thread owns the pairs (k, M-k), k = j + m T < M/2 (thread 0's first pair is (0, M/2)).
        // Z'[k] is its own stage-0 register m; Z'[M-k] belongs to thread T-j and travels through smem.
        float2 xb[R / 2];
        if constexpr (RDIRECT)
        {
#pragma unroll
            for (int m = 0; m < R / 2; ++m)
            {
                const int plo = upg.real_lo (m), phi = (m == 0 && j == 0) ? W_HALF_ROW<LOGW>() : upg.real_hi (m);
                v[m] = make_float2 (__ldg (in + plo), __ldg (in + plo + WL));
                xb[m] = make_float2 (__ldg (in + phi), __ldg (in + phi + WL));
            }
        }
        else if constexpr (UNORD)
        {
            if constexpr (! IN_STAGED)
            {
                staging_fill<G> (sf, in, j, logW, active);
                tsync<T, WS>();
            }
#pragma unroll
            for (int m = 0; m < R / 2; ++m)
            {
                v[m] = staged_load (sf, up.real_lo (m), WL);
                xb[m] = staged_load (sf, (m == 0 && j == 0) ? W_HALF_ROW<LOGW>() : up.real_hi (m), WL);
            }
            if constexpr (! SHFL_MIRROR)
                tsync<T, WS>(); // staging image fully consumed before the natural-order image overwrites it
        }
        else
        {
            if constexpr (IN_UNION != 0)
            {
                // ordered spectrum already in shared memory (`su`, natural order, unpadded): unit-stride reads both ways
                static_assert (IN_UNION == 0 || FMT == 0, "landing-buffer input is for the pffft packing");
                const float2* lo = su + j;
                const float2* hi = su + (M - T) - j;
#pragma unroll
                for (int m = 0; m < R / 2; ++m)
                {
                    const float2* ph = (m == 0 && j == 0) ? su + M / 2 : hi - m * T + T;
                    v[m] = lds2 (lo + m * T);
                    xb[m] = lds2 (ph);
                }
                smem_was_read = true;
            }
            else
            {
                const float2* __restrict__ lo = reinterpret_cast<const float2*> (in) + j;
                const float2* __restrict__ hi = reinterpret_cast<const float2*> (in) + (M - T) - j;
#pragma unroll
                for (int m = 0; m < R / 2; ++m)
                {
                    const float2* ph = (m == 0 && j == 0) ? reinterpret_cast<const float2*> (in) + M / 2 : hi - m * T + T;
                    v[m] = ldg_in<T> (lo + m * T);
                    xb[m] = ldg_in<T> (ph);
                }
                if (FMT == 1 && j == 0)
                    v[0].y = ldg_stream (reinterpret_cast<const float2*> (in) + M).x; // Nyquist lives in bin M, not in float 1
            }
        }
        const float2 wj = __ldg (a.rtw + j);
#pragma unroll
        for (int m = 0; m < R / 2; ++m)
        {
            const float2 xa = v[m], xm = xb[m];
            const float2 wh = real_tw<R, RTW_DERIVE> (wj, a.rtw + j + m * T, m);                         // w_k / 2
            const float2 cm = make_float2 (xm.x, -xm.y);                   // conj X[M-k]
            const float2 e = f2_add (xa, cm), d = f2_sub (xa, cm);
            const float2 wd = cmul_dir<+1> (d, wh);                        // conj(w_k) d / 2
            const float2 two = make_float2 (2.f, 2.f);
            float2 zk = f2_fma (make_float2 (-wd.y, wd.x), two, e);                      // e + i conj(w) d
            float2 zm = f2_fma (make_float2 (wd.y, wd.x), two, make_float2 (e.x, -e.y)); // conj(e - i conj(w) d)
            int slot = mirror_slot<G> (j, m);
            if (m == 0 && j == 0)
            {
                zk = make_float2 (xa.x + xa.y, xa.x - xa.y);   // Z'[0] from (DC, Nyquist)
                zm = make_float2 (2.f * xm.x, -2.f * xm.y);    // Z'[M/2] = 2 conj X[M/2]
                slot = G::pad (M / 2);
            }
            v[m] = zk;
            if constexpr (SHFL_MIRROR)
                xb[m] = zm;
            else
                sts2 (s + slot, zm);
        }
        if constexpr (SHFL_MIRROR)
        {
            // Z'[M-k] computed by thread T-j is this thread's register R-1-m; thread 0 computed its own registers R-m
            // (bins M - m T) and, as its first pair, R/2 (bin M/2)
#pragma unroll
            for (int m = 0; m < R / 2; ++m)
                v[R - 1 - m] = shfl2 (xb[m], (T - j) & (T - 1), T);
            if (j == 0)
            {
#pragma unroll
                for (int m = 1; m < R / 2; ++m)
                    v[R - m] = xb[m];
                v[R / 2] = xb[0];
            }
            if constexpr (UNORD && ! RDIRECT)
                smem_was_read = true; // the staging image was read: a barrier must precede the first exchange
        }
        else
        {
            static_assert (SHFL_MIRROR || IN_UNION == 0, "landing-buffer C2R input needs the shuffle merge (the exchange buffer is not synchronised yet)");
            tsync<T, WS>();
            gather_natural<G, R / 2, R> (v, j, s);
            smem_was_read = true;
        }
    }

    // ---- the stages -----------------------------------------------------------------------------
    Stages<G, DIR, 0, WS, IN_UNION == 1>::run (v, j, s, a.tw, smem_was_read, input_consumed, last_gathered);
    if (G::S > 1)
        smem_was_read = true;

    // ---- epilogue -------------------------------------------------------------------------------
    if constexpr (OUT_REGS)
    {
        static_assert (! OUT_REGS || KIND == C2C_BWD || KIND == C2R, "OUT_REGS is for the inverse kinds");
#pragma unroll
        for (int m = 0; m < R; ++m)
            vout[m] = v[m];
    }
    else if constexpr (KIND == C2C_BWD || KIND == C2R || (KIND == C2C_FWD && ! UNORD))
    {
        if (active)
        {
            float2* __restrict__ out2 = reinterpret_cast<float2*> (out) + j;
            constexpr float inv_n = 1.f / (float) (KIND == C2R ? 2 * M : M);
#pragma unroll
            for (int m = (HALF_OUT ? R / 2 : 0); m < R; ++m)
                out2[m * T] = (FMT == 1 && KIND != C2C_FWD) ? f2_mul (v[m], make_float2 (inv_n, inv_n)) : v[m];
        }
    }
    else if constexpr (KIND == C2C_FWD && UDIRECT && ! OUT_STAGED)
    {
        float* __restrict__ ob = out + u_base;
#pragma unroll
        for (int m = 0; m < R; ++m)
        {
            const float recv = shfl1 (u_odd ? v[m].x : v[m].y, (j ^ 1) & (SW - 1), SW);
            const float2 o = u_odd ? make_float2 (recv, v[m].y) : make_float2 (v[m].x, recv);
            if (active)
                *reinterpret_cast<float2*> (ob + (m % ULT) * (T / UW) * 2 * UW * UW + (m / ULT) * 2 * UW) = o;
        }
    }
    else if constexpr (KIND == C2C_FWD)
    {
        if (smem_was_read)
            tsync<T, WS>();
#pragma unroll
        for (int m = 0; m < R; ++m)
            staged_store (sf, up.cplx (m), WL, v[m]);
        tsync<T, WS>();
        if constexpr (! OUT_STAGED)
            staging_drain<G> (sf, out, j, logW, active);
    }
    else // R2C: split step  X[k] = E - i w_k D,  X[M-k] = conj(E + i w_k D),  E,D = (Z[k] +- Z*[M-k]) / 2
    {
        // Z[k], k = j + m T < M/2, is this thread's register m; Z[M-k] is register R-1-m of thread T-j:
        // only the upper half of the spectrum goes through shared memory.
        float2 zb[R / 2];
        if constexpr (SHFL_MIRROR)
        {
            // transforms that live inside one warp: the mirror element comes straight from thread T-j's register
            // R-1-m by shuffle (half the shared-memory wavefronts of the store + load round trip, no barriers);
            // thread 0's mirrors are its own registers R-m (bins M - m T) and R/2 (bin M/2)
#pragma unroll
            for (int m = 0; m < R / 2; ++m)
                zb[m] = shfl2 (v[R - 1 - m], (T - j) & (T - 1), T);
            if (j == 0)
            {
#pragma unroll
                for (int m = 1; m < R / 2; ++m)
                    zb[m] = v[R - m];
                zb[0] = v[R / 2];
            }
            if constexpr (UNORD && ! RDIRECT)
                if (smem_was_read)
                    tsync<T, WS && ! (IN_UNION == 1 && G::S == 1)>(); // the last exchange has been read: the staging image may overwrite it
        }
        else
        {
            if (smem_was_read)
                tsync<T, WS && ! (IN_UNION == 1 && G::S == 1)>();
            scatter_natural<G, R / 2, R> (v, j, s);
            tsync<T, WS>();
#pragma unroll
            for (int m = 0; m < R / 2; ++m)
                zb[m] = lds2 (s + ((m == 0 && j == 0) ? G::pad (M / 2) : mirror_slot<G> (j, m)));
            if constexpr (UNORD && ! RDIRECT)
                tsync<T, WS>(); // natural-order image fully consumed before the staging image overwrites it
        }
        const float2 wj = __ldg (a.rtw + j);
        float2* __restrict__ lo = reinterpret_cast<float2*> (out) + j;
        float2* __restrict__ hi = reinterpret_cast<float2*> (out) + (M - T) - j;
#pragma unroll
        for (int m = 0; m < R / 2; ++m)
        {
            const float2 za = v[m], zm = zb[m];
            const float2 wh = real_tw<R, RTW_DERIVE> (wj, a.rtw + j + m * T, m);                         // w_k / 2
            const float2 cm = make_float2 (zm.x, -zm.y);                   // conj Z[M-k]
            const float2 e = f2_add (za, cm), d = f2_sub (za, cm);         // 2E, 2D
            const float2 wd = cmul_dir<-1> (d, wh);                        // w_k D
            float2 xa = f2_fma (e, make_float2 (0.5f, 0.5f), make_float2 (wd.y, -wd.x));    // E - i w D
            float2 xm = f2_fma (e, make_float2 (0.5f, -0.5f), make_float2 (-wd.y, -wd.x));  // conj(E + i w D)
            const bool special = (m == 0 && j == 0);
            if (special)
            {
                xa = make_float2 (za.x + za.y, za.x - za.y); // (DC, Nyquist)
                xm = make_float2 (zm.x, -zm.y);              // X[M/2] = conj Z[M/2]
            }
            if constexpr (RDIRECT)
            {
                if (active)
                {
                    const int plo = upg.real_lo (m), phi = special ? W_HALF_ROW<LOGW>() : upg.real_hi (m);
                    out[plo] = xa.x;
                    out[plo + WL] = xa.y;
                    out[phi] = xm.x;
                    out[phi + WL] = xm.y;
                }
            }
            else if constexpr (UNORD)
            {
                staged_store (sf, up.real_lo (m), WL, xa);
                staged_store (sf, special ? W_HALF_ROW<LOGW>() : up.real_hi (m), WL, xm);
            }
            else if (active)
            {
                if (FMT == 1 && special)
                {
                    reinterpret_cast<float2*> (out)[M] = make_float2 (xa.y, 0.f); // Nyquist as bin M
                    xa.y = 0.f;
                }
                lo[m * T] = xa;
                float2* ph = special ? reinterpret_cast<float2*> (out) + M / 2 : hi - m * T + T;
                *ph = xm;
            }
        }
        if constexpr (UNORD && ! RDIRECT)
        {
            tsync<T, WS>();
            if constexpr (! OUT_STAGED)
                staging_drain<G> (sf, out, j, logW, active);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// the batched transform kernel.  blockDim.x = T * (transforms per CTA); dynamic smem = transforms per
// CTA * SMEM_F2 * 8 bytes.
// ---------------------------------------------------------------------------------------------
template <int LOGM, int R, int KIND, int LOGW, int FMT = 0>
FFT_HD void fft_body (const FftArgs& a)
{
    using G = Geo<LOGM, R>;
    constexpr int T = G::T;
    constexpr int SMEM_F2 = LOGW != 0 ? G::SMEM_F2_UNORD : G::SMEM_F2;
    FFT_DYN_SMEM (float2, smem);

    const int tid = (int) threadIdx.x;
    const int j = tid & (T - 1);
    const int lt = tid / T;
    const int per_cta = (int) blockDim.x / T;
    const long long x = (long long) blockIdx.x * per_cta + lt;
    const bool active = x < a.batch;

    // CTAs past the end of the batch re-read the last transform (loads stay unpredicated) and skip stores
    const unsigned xc = active ? (unsigned) x : (unsigned) a.batch - 1u;
    unsigned xo = 0, xi = xc;
    if (a.inner < a.batch) // two-level batch (STFT gather); plain batches skip the division
    {
        xo = xc / (unsigned) a.inner;
        xi = xc - xo * (unsigned) a.inner;
    }
    const float* in = a.in + (long long) xo * a.in_outer + (long long) xi * a.in_inner;
    float* out = a.out + (long long) xo * a.out_outer + (long long) xi * a.out_inner;
    if (a.pf_ahead > 0)
    {
        const long long xn = x + (long long) a.pf_ahead * per_cta;
        if (xn < a.batch)
        {
            unsigned no = 0, ni = (unsigned) xn;
            if (a.inner < a.batch)
            {
                no = ni / (unsigned) a.inner;
                ni -= no * (unsigned) a.inner;
            }
            prefetch_transform_l2<G> (a.in + (long long) no * a.in_outer + (long long) ni * a.in_inner, j);
        }
    }
    fft_core<LOGM, R, KIND, LOGW, false, false, false, false, NoHook, false, FMT> (in, out, active, j, smem + lt * SMEM_F2, a.tw, a.rtw);
}

// threads per CTA / occupancy targets
template <int LOGM, int R>
struct Launch
{
    using G = Geo<LOGM, R>;
    static constexpr int THREADS = G::T >= 256 ? G::T : 256;
    static constexpr int PER_CTA = THREADS / G::T;
    static constexpr int SMEM_BYTES = PER_CTA * G::SMEM_F2 * 8;
    static constexpr int SMEM_BYTES_UNORD = PER_CTA * G::SMEM_F2_UNORD * 8;
    // R = 16 kernels fit 64 registers per thread (1024 resident threads per SM), R = 32 kernels need 128 (512)
    static constexpr int MIN_BLOCKS = (R == 16 ? 1024 : 512) / THREADS < 1 ? 1 : (R == 16 ? 1024 : 512) / THREADS;
};

template <int LOGM, int R, int KIND, int LOGW>
__global__ void __launch_bounds__ (Launch<LOGM, R>::THREADS, Launch<LOGM, R>::MIN_BLOCKS) fft_kernel (const FftArgs a)
{
    fft_body<LOGM, R, KIND, LOGW> (a);
}
// ---------------------------------------------------------------------------------------------
// Dense batches of TINY transforms (16 .. 64 complex points: one, two or four threads per transform).  In fft_kernel a load
// instruction of such a transform covers 8 .. 32 bytes of every 128-byte line it touches, so a warp's access spreads over 8 .. 32
// lines: sector-efficient at best, but four to sixteen times the L1 tag work and, for one or two threads per transform, partial-
// sector stores (ncu: l1tex-bound at 1.8 .. 5.3 TB/s).  Here the CTA's transforms, which are contiguous in a dense batch, are copied
// with fully coalesced 64-bit accesses into padded shared-memory rows (the pad spreads a warp's transforms over the banks), every
// transform runs fft_core on its row (input = private shared-memory image, output = the same row through a generic pointer) and the
// rows go back with coalesced stores (unordered inputs are copied straight into the transforms' staging images instead).  Batch
// stride = transform length on both sides, 16 / 32 complex points; everything else keeps fft_kernel.
// ---------------------------------------------------------------------------------------------
template <int LOGM, int KIND, int LOGW>
struct SmallLaunch
{
    using G = Geo<LOGM, 16>;
    using L = Launch<LOGM, 16>;
    // float2 slots between rows: a half-warp's rows start 8 / 4 / 2 banks apart for 4 / 2 / 1 threads per transform (one thread per
    // transform with an unordered output keeps rows 16-byte aligned for the 128-bit drain and accepts two-way conflicts)
    static constexpr int PAD = G::T >= 4 ? 4 : G::T == 2 ? 2 : (LOGW != 0 ? 2 : 1);
    static constexpr int PITCH = G::M + PAD;
    static constexpr int XCH_F2 = LOGW != 0 ? G::SMEM_F2_UNORD : G::SMEM_F2;
    static constexpr int SMEM_BYTES = L::PER_CTA * (PITCH + XCH_F2) * 8;
    // unordered INPUTS (inverse kinds) are copied straight into the padded staging image fft_core expects (IN_STAGED)
    static constexpr bool IN_IMAGE = LOGW != 0 && (KIND == C2C_BWD || KIND == C2R);
    // one or two threads per transform: 3.1-3.3x / 1.5-1.6x over fft_kernel on B200; with four (64 points) it is a tie for ordered
    // data and 13-17 % slower for unordered outputs (profiles/r02_small_kernel.txt), so those stay with fft_kernel
    static constexpr bool APPLIES = G::T <= 2;
};
template <int LOGM, int KIND, int LOGW>
FFT_HD void small_body (const FftArgs& a)
{
    using SL = SmallLaunch<LOGM, KIND, LOGW>;
    using G = typename SL::G;
    constexpr int T = G::T, M = G::M, PER_CTA = SL::L::PER_CTA, THREADS = SL::L::THREADS, PITCH = SL::PITCH;
    constexpr int ITERS = PER_CTA * M / THREADS; // = 16
    FFT_DYN_SMEM (float2, smem);
    float2* rows = smem;
    float2* xch = smem + PER_CTA * PITCH;
    const int tid = (int) threadIdx.x;
    const long long x0 = (long long) blockIdx.x * PER_CTA;
    const long long left = (long long) a.batch - x0;
    const int total = (int) (left < PER_CTA ? left : PER_CTA) * M; // complex elements of this CTA's transforms
    const float2* __restrict__ in2 = reinterpret_cast<const float2*> (a.in) + x0 * M;
    float2* __restrict__ out2 = reinterpret_cast<float2*> (a.out) + x0 * M;
    float2 t[ITERS];
    const int j = tid & (T - 1), lt = tid / T;
    float2* row = rows + lt * PITCH;
    if constexpr (SL::IN_IMAGE)
    {
        // unordered input: 128-bit coalesced copy of the CTA's spectra into every transform's staging image (the layout staging_fill builds)
        const float4* __restrict__ in4 = reinterpret_cast<const float4*> (a.in) + x0 * (M / 2);
        float4 t4[ITERS / 2];
#pragma unroll
        for (int i = 0; i < ITERS / 2; ++i)
        {
            const int e = tid + i * THREADS;
            t4[i] = e < total / 2 ? ldg_stream (in4 + e) : make_float4 (0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int i = 0; i < ITERS / 2; ++i)
        {
            const int e = tid + i * THREADS;
            sts4 (reinterpret_cast<float*> (xch + (e >> (LOGM - 1)) * SL::XCH_F2) + upad (4 * (e & (M / 2 - 1)), LOGW), t4[i]);
        }
        __syncthreads();
        fft_core<LOGM, 16, KIND, LOGW, true, false, false, 0> (nullptr, reinterpret_cast<float*> (row), true, j, xch + lt * SL::XCH_F2, a.tw, a.rtw);
    }
    else
    {
#pragma unroll
        for (int i = 0; i < ITERS; ++i)
        {
            const int e = tid + i * THREADS;
            t[i] = e < total ? ldg_stream (in2 + e) : make_float2 (0.f, 0.f);
        }
#pragma unroll
        for (int i = 0; i < ITERS; ++i)
        {
            const int e = tid + i * THREADS;
            sts2 (rows + (e >> LOGM) * PITCH + (e & (M - 1)), t[i]);
        }
        __syncthreads();
        fft_core<LOGM, 16, KIND, LOGW, false, false, false, 2> (nullptr, reinterpret_cast<float*> (row), true, j, xch + lt * SL::XCH_F2, a.tw, a.rtw, row);
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < ITERS; ++i)
    {
        const int e = tid + i * THREADS;
        t[i] = lds2 (rows + (e >> LOGM) * PITCH + (e & (M - 1)));
    }
#pragma unroll
    for (int i = 0; i < ITERS; ++i)
    {
        const int e = tid + i * THREADS;
        if (e < total)
            out2[e] = t[i];
    }
}
template <int LOGM, int KIND, int LOGW>
__global__ void __launch_bounds__ (Launch<LOGM, 16>::THREADS, 3) fft_small_kernel (const FftArgs a)
{
    small_body<LOGM, KIND, LOGW> (a);
}

// the same transform with the JUCE adapter's conventions (fft_core: FMT = 1), ordered layouts, R2C / C2R / C2C_BWD
template <int LOGM, int R, int KIND>
__global__ void __launch_bounds__ (Launch<LOGM, R>::THREADS, Launch<LOGM, R>::MIN_BLOCKS) fft_kernel_juce (const FftArgs a)
{
    fft_body<LOGM, R, KIND, 0, 1> (a);
}

// ---------------------------------------------------------------------------------------------
// Frame-gather (STFT analysis) kernel: R2C of OVERLAPPING windows of one signal, times an optional analysis
// window.  A CTA owns PER_CTA consecutive frames of one channel.  Grid = outer * groups, groups =
// ceil (inner / PER_CTA).
//   UNION = false: every transform loads its own frame straight into registers (re-reads of the overlap are
//                  L2 hits) -- the faster variant on B200: the kernel is bound by the L1/shared-memory pipe,
//                  not by L2->SM bytes (ncu: l1tex 84 %, DRAM 47 %), and staging costs extra wavefronts.
//   UNION = true : the union of the CTA's frames ((PER_CTA-1) hop + N floats instead of PER_CTA N) is copied
//                  into shared memory once with linear 128-bit loads and every transform takes its stage-0
//                  registers from there; 2.3x fewer L2->SM bytes at hop = N/4 (kept selectable for parts where
//                  that is the bound).  Needs 0 < in_inner <= N.
// in_inner and in_outer must be even (8-byte aligned frames).
// ---------------------------------------------------------------------------------------------
template <int LOGM, int R, int LOGW, bool UNION>
FFT_HD void stft_body (const FftArgs& a)
{
    using G = Geo<LOGM, R>;
    constexpr int T = G::T, NFL = 2 * G::M;
    constexpr int SMEM_F2 = LOGW != 0 ? G::SMEM_F2_UNORD : G::SMEM_F2;
    FFT_DYN_SMEM (float2, smem);

    const int tid = (int) threadIdx.x;
    const int j = tid & (T - 1);
    const int lt = tid / T;
    const int per_cta = (int) blockDim.x / T;
    const int o = (int) blockIdx.x / a.groups;
    const int g = (int) blockIdx.x - o * a.groups;
    const int f0 = g * per_cta;
    const int nact = a.inner - f0 < per_cta ? a.inner - f0 : per_cta;
    const bool active = lt < nact;
    const int ltc = active ? lt : nact - 1; // idle transforms of the last group redo its last frame and skip the store

    const float* __restrict__ base = a.in + (long long) o * a.in_outer + (long long) f0 * a.in_inner;
    float* out = a.out + (long long) o * a.out_outer + (long long) (f0 + ltc) * a.out_inner;
    if (a.pf_ahead > 0)
    {
        const long long bn = (long long) blockIdx.x + a.pf_ahead;
        const long long on = bn / a.groups;
        const long long fn = (bn - on * a.groups) * per_cta + lt;
        if (on * a.inner < a.batch && fn < a.inner)
            prefetch_transform_l2<G> (a.in + on * a.in_outer + fn * a.in_inner, j);
    }
    if constexpr (! UNION)
    {
        fft_core<LOGM, R, R2C, LOGW, false, false, false, false> (base + (long long) ltc * a.in_inner, out, active, j, smem + lt * SMEM_F2, a.tw, a.rtw,
                                                                  nullptr, reinterpret_cast<const float2*> (a.window));
        return;
    }
    const int span = (nact - 1) * (int) a.in_inner + NFL; // floats, <= per_cta * NFL
    float* su = reinterpret_cast<float*> (smem);
    if (a.vec4)
    {
        for (int i = tid; i - tid < span / 4; i += (int) blockDim.x)
        {
            if (i < span / 4)
                sts4 (su + 4 * i, ldg_stream (reinterpret_cast<const float4*> (base) + i));
            else
                smem_skip();
        }
    }
    else
    {
        for (int i = tid; i - tid < span / 2; i += (int) blockDim.x)
        {
            if (i < span / 2)
                sts2 (smem + i, ldg_stream (reinterpret_cast<const float2*> (base) + i));
            else
                smem_skip();
        }
    }
    __syncthreads();
    fft_core<LOGM, R, R2C, LOGW, false, false, false, true> (nullptr, out, active, j, smem + lt * SMEM_F2, a.tw, a.rtw,
                                                             smem + ltc * (int) (a.in_inner / 2), reinterpret_cast<const float2*> (a.window));
}

template <int LOGM, int R, int LOGW, bool UNION>
__global__ void __launch_bounds__ (Launch<LOGM, R>::THREADS, Launch<LOGM, R>::MIN_BLOCKS) stft_kernel (const FftArgs a)
{
    stft_body<LOGM, R, LOGW, UNION> (a);
}

// ---------------------------------------------------------------------------------------------
// Overlap-add synthesis (inverse STFT): C2R of the frames of a channel, optional synthesis window, frames summed at
// hop distance into the output signal -- one kernel, owner-computes, no atomics:
//   out[c][t] = scale * sum over frames f with 0 <= t - f hop < N of  window[t - f hop] * C2R (spectrum (c, f)) [t - f hop]
// A CTA owns the frames [fs, fe) of one channel (a "segment") and walks through them PER_CTA at a time: every
// transform leaves its windowed frame in its own shared-memory region; the CTA then sums the frames over the span
// they cover plus the tail carried from the previous group, stores the PER_CTA * hop samples that are final and keeps
// the remaining N - hop as the next tail.  Segments other than a channel's first start ceil (N / hop) - 1 frames early
// (halo, recomputed, not stored) so that segments never need each other's partial sums.  This is the step the
// reference leaves to the caller around fft_transform (BACKWARD) + fft_accumulate (chowdsp_fft.h:138,160;
// test/test.cpp:214-218); fusing it removes the write + re-read of every frame (N / hop times the signal).
// Grid = channels * nseg.  Needs 0 < hop <= N; the input frames are ordered or unordered spectra.
// Shared memory: [PER_CTA exchange / frame buffers][2 tails of N - hop floats].
// ---------------------------------------------------------------------------------------------
// One overlap-add pass: out sample s = tail[s] + sum over the frames g < nact that cover it of frame_g[s - g hop].
// Every thread owns the samples s = VEC (tid + k nthreads) .. + VEC, so no two threads touch the same sum; frames
// are tried in order (nact <= 16 compares per sample group, no division).  Samples below `done` are final and go
// to global memory (from first_owned on), the others become the next tail (or, at the end of a channel, output).
template <int VEC>
FFT_HD void ola_pass (const float* frames, int frame_stride, int nfl, int hop, int nact, int span, int done, int tail_n,
                      const float* tail_cur, float* tail_new, float* __restrict__ sig, long long first_owned, bool keep_tail, int tid, int nthreads)
{
    for (int s = tid * VEC; s < span; s += nthreads * VEC)
    {
        float acc[VEC];
        if (s < tail_n)
        {
            if constexpr (VEC == 4)
            {
                const float4 t = lds4 (tail_cur + s);
                acc[0] = t.x; acc[1] = t.y; acc[2] = t.z; acc[3] = t.w;
            }
            else
                acc[0] = lds1 (tail_cur + s);
        }
        else
        {
#pragma unroll
            for (int i = 0; i < VEC; ++i)
                acc[i] = 0.f;
        }
#pragma unroll 4
        for (int g = 0; g < nact; ++g)
        {
            const int n = s - g * hop;
            if ((unsigned) n < (unsigned) nfl)
            {
                if constexpr (VEC == 4)
                {
                    const float4 x = lds4 (frames + g * frame_stride + n);
                    acc[0] += x.x; acc[1] += x.y; acc[2] += x.z; acc[3] += x.w;
                }
                else
                    acc[0] += lds1 (frames + g * frame_stride + n);
            }
        }
        if (s < done || ! keep_tail)
        {
            if (s >= first_owned)
            {
                if constexpr (VEC == 4)
                    *reinterpret_cast<float4*> (sig + s) = make_float4 (acc[0], acc[1], acc[2], acc[3]);
                else
                    sig[s] = acc[0];
            }
        }
        else
        {
            if constexpr (VEC == 4)
                sts4 (tail_new + (s - done), make_float4 (acc[0], acc[1], acc[2], acc[3]));
            else
                sts1 (tail_new + (s - done), acc[0]);
        }
    }
}

template <int LOGM, int R, int LOGW>
FFT_HD void istft_body (const FftArgs& a)
{
    using G = Geo<LOGM, R>;
    constexpr int T = G::T, NFL = 2 * G::M;
    constexpr int SMEM_F2 = LOGW != 0 ? G::SMEM_F2_UNORD : G::SMEM_F2;
    FFT_DYN_SMEM (float2, smem);

    const int tid = (int) threadIdx.x, nthreads = (int) blockDim.x;
    const int j = tid & (T - 1);
    const int lt = tid / T;
    const int per_cta = nthreads / T;
    const int hop = (int) a.out_inner, frames = a.inner;
    const int tail_n = NFL - hop;                           // samples carried between groups
    float* tail0 = reinterpret_cast<float*> (smem + per_cta * SMEM_F2);
    float* tail1 = tail0 + ((tail_n + 3) & ~3);
    float2* fb = smem + lt * SMEM_F2;                       // this transform's exchange region, then its frame

    const int c = (int) blockIdx.x / a.nseg;
    const int seg = (int) blockIdx.x - c * a.nseg;
    const int fs = seg * a.seg_frames;
    const int fe = fs + a.seg_frames < frames ? fs + a.seg_frames : frames;
    const int halo = (NFL + hop - 1) / hop - 1;
    const int f_begin = fs - halo > 0 ? fs - halo : 0;
    const long long own_start = (long long) fs * hop;       // first sample this CTA stores
    const bool last_seg = fe == frames;
    const float* __restrict__ spec = a.in + (long long) c * a.in_outer;
    float* __restrict__ sig = a.out + (long long) c * a.out_outer;
    const float2* __restrict__ win2 = reinterpret_cast<const float2*> (a.window);

    for (int i = tid; i < tail_n; i += nthreads)
        tail0[i] = 0.f;
    float* tail_cur = tail0;
    float* tail_new = tail1;
    for (int f0 = f_begin; f0 < fe; f0 += per_cta)
    {
        const int nact = fe - f0 < per_cta ? fe - f0 : per_cta;
        const int ltc = lt < nact ? lt : nact - 1;          // idle transforms redo the group's last frame; it is never summed
        float2 v[R];
        fft_core<LOGM, R, C2R, LOGW, false, false, false, false, NoHook, true> (spec + (long long) (f0 + ltc) * a.in_inner, nullptr, true, j, fb, a.tw, a.rtw,
                                                                               nullptr, nullptr, NoHook(), v);
        tsync<T, true>(); // the transform's last exchange has been read: its region becomes the frame buffer
#pragma unroll
        for (int m = 0; m < R; ++m)
        {
            float2 x = f2_mul (v[m], make_float2 (a.scale, a.scale));
            if (win2 != nullptr)
                x = f2_mul (x, __ldg (win2 + j + m * T));
            sts2 (fb + j + m * T, x);
        }
        __syncthreads();
        // ---- overlap-add over the span of this group; sample index s is relative to the group's first frame ----
        const int span = (nact - 1) * hop + NFL, done = nact * hop;
        const long long t0 = (long long) f0 * hop;
        const bool keep_tail = ! (last_seg && f0 + nact == fe); // at the end of the channel the tail is output too
        if (a.vec4)
            ola_pass<4> (reinterpret_cast<const float*> (smem), SMEM_F2 * 2, NFL, hop, nact, span, done, tail_n, tail_cur, tail_new,
                         sig + t0, own_start - t0, keep_tail, tid, nthreads);
        else
            ola_pass<1> (reinterpret_cast<const float*> (smem), SMEM_F2 * 2, NFL, hop, nact, span, done, tail_n, tail_cur, tail_new,
                         sig + t0, own_start - t0, keep_tail, tid, nthreads);
        __syncthreads();
        float* sw = tail_cur;
        tail_cur = tail_new;
        tail_new = sw;
    }
}

// ---------------------------------------------------------------------------------------------
// Overlap-add synthesis with the sums in REGISTERS (ristft_kernel): hop = N / 2, N / 4 or N / 8, transforms of 32 .. 256 threads
// (N = 1024 .. 8192), ordered or unordered spectra.  Thread j's result registers are the sample pairs j + m T, and hop / 2 = T HQ
// pairs, so slot m of a frame is slot m - HQ of the next one: the N - hop samples a frame shares with its successors stay in
// R - HQ accumulator registers of the same thread that shift by HQ per frame, the hop samples that are final leave straight from
// registers -- the scheme of the warp-pipelined wistft_kernel, for any transform whose threads are whole warps.  A transform's
// thread group walks through the frames of one (channel, segment) item; no shared-memory frame buffers, no carried tails, no CTA
// barrier (istft_kernel rewrites a tail of N - hop samples in shared memory for every group of 1 .. 8 frames: 1.7 .. 2.9 TB/s at
// these sizes, tools/stft_sweep.py).  Segments other than a channel's first recompute a halo of N / hop - 1 frames.
// a.in_inner / in_outer: floats between frames / channels of the spectra; a.out_inner = hop; a.out_outer: floats between channels
// of the signal; a.nseg, a.seg_frames: segments per channel and frames per segment; a.scale; a.window (N floats or nullptr).
// CARRY (streaming synthesis, fft_stft_stream_synthesize): one item per channel (a.nseg = 1, a.seg_frames = a.inner) and no halo;
// the accumulators start from, and end in, `carry` + c (N - hop) / 2: the N - hop samples after the call's last hop, as float2
// [i][j] (sample pair i T + j of the carried span, so the load and the store are coalesced).  The sums are formed in the same
// order as in one unsegmented run, so the signal does not depend on how the frames are split into calls.
// ---------------------------------------------------------------------------------------------
template <int LOGM, int HQ, int LOGW, bool CARRY = false>
FFT_HD void ristft_body (const FftArgs& a, float2* __restrict__ carry = nullptr)
{
    constexpr int R = 16;
    using G = Geo<LOGM, R>;
    constexpr int T = G::T;
    static_assert (HQ >= 1 && 2 * HQ <= R && R % HQ == 0, "hop = N/2, N/4 or N/8");
    // transforms smaller than a warp share their warp-level barriers with their neighbours: every item then runs the same number of
    // iterations (seg_frames + HALO; frames outside its range are computed on a clamped index and neither summed nor stored)
    constexpr bool UNIFORM = T < 32;
    constexpr int NACC = R - HQ, HOP2 = T * HQ, HALO = R / HQ - 1;
    constexpr int SMEM_F2 = LOGW != 0 ? G::SMEM_F2_UNORD : G::SMEM_F2;
    FFT_DYN_SMEM (float2, smem);
    const int tid = (int) threadIdx.x;
    const int j = tid & (T - 1), lt = tid / T, per_cta = (int) blockDim.x / T;
    float2* fb = smem + lt * SMEM_F2;
    const int frames = a.inner;
    const long long items = (long long) (a.batch / a.inner) * a.nseg;
    long long item = (long long) blockIdx.x * per_cta + lt;
    const bool item_ok = item < items;
    if (! item_ok)
    {
        if constexpr (! UNIFORM)
            return; // every barrier below is private to the transform's own warps
        item = items - 1;
    }
    const int c = (int) (item / a.nseg);
    const int fs = (int) (item - (long long) c * a.nseg) * a.seg_frames;
    const int fe = fs + a.seg_frames < frames ? fs + a.seg_frames : frames;
    const float* __restrict__ spec = a.in + (long long) c * a.in_outer;
    float2* __restrict__ sig2 = reinterpret_cast<float2*> (a.out + (long long) c * a.out_outer) + j;
    const float2* __restrict__ win2 = reinterpret_cast<const float2*> (a.window);
    const float2 scale2 = make_float2 (a.scale, a.scale);
    float2 acc[NACC];
    float2* __restrict__ st = CARRY ? carry + (long long) c * (NACC * T) + j : nullptr;
#pragma unroll
    for (int i = 0; i < NACC; ++i)
        acc[i] = CARRY ? st[i * T] : make_float2 (0.f, 0.f);
    const int f_first = CARRY ? fs : UNIFORM ? fs - HALO : (fs - HALO > 0 ? fs - HALO : 0);
    const int f_last = UNIFORM ? fs + a.seg_frames : fe;
    for (int ff = f_first; ff < f_last; ++ff)
    {
        const bool valid = ! UNIFORM || (item_ok && ff >= 0 && ff < fe);
        const int f = valid ? ff : (fe - 1);
#ifndef CFB_RISTFT_NO_PREFETCH
        // the frames of an item are transformed strictly one after the other: ask L2 for the next one now (one line per thread)
        if (ff + 1 < fe && ff + 1 >= 0)
            prefetch_transform_l2<G> (spec + (long long) (ff + 1) * a.in_inner, j);
#endif
        float2 v[R];
        fft_core<LOGM, R, C2R, LOGW, false, false, false, 0, NoHook, true> (spec + (long long) f * a.in_inner, nullptr, true, j, fb, a.tw, a.rtw, nullptr, nullptr, NoHook(), v);
        tsync<T, true>(); // the last exchange has been read by every thread of the transform: the next frame may write the region
        if (! valid)
            continue;
#pragma unroll
        for (int m = 0; m < R; ++m)
        {
            v[m] = f2_mul (v[m], scale2);
            if (win2 != nullptr)
                v[m] = f2_mul (v[m], __ldg (win2 + j + m * T));
        }
        float2* __restrict__ o = sig2 + (long long) f * HOP2;
        if (f >= fs)
        {
#pragma unroll
            for (int m = 0; m < HQ; ++m)
                o[m * T] = f2_add (acc[m], v[m]);
        }
#pragma unroll
        for (int i = 0; i < NACC; ++i)
            acc[i] = i + HQ < NACC ? f2_add (acc[i + HQ], v[i + HQ]) : v[i + HQ];
        if (! CARRY && f + 1 == fe && fe == frames) // end of the channel: the carried samples are output too
        {
#pragma unroll
            for (int i = 0; i < NACC; ++i)
                o[HOP2 + T * i] = acc[i];
        }
    }
    if (CARRY && item_ok)
    {
#pragma unroll
        for (int i = 0; i < NACC; ++i)
            st[i * T] = acc[i];
    }
}
#ifndef CFB_RISTFT_MINB
#define CFB_RISTFT_MINB 2 // A/B switch (tools/ only): resident CTAs per SM the register budget of ristft_kernel is sized for
#endif
template <int LOGM, int HQ, int LOGW>
__global__ void __launch_bounds__ (Launch<LOGM, 16>::THREADS, CFB_RISTFT_MINB) ristft_kernel (const FftArgs a)
{
    ristft_body<LOGM, HQ, LOGW> (a);
}
template <int LOGM, int HQ, int LOGW>
__global__ void __launch_bounds__ (Launch<LOGM, 16>::THREADS, CFB_RISTFT_MINB) ristft_carry_kernel (const FftArgs a, float2* carry)
{
    ristft_body<LOGM, HQ, LOGW, true> (a, carry);
}

template <int LOGM, int R, int LOGW>
__global__ void __launch_bounds__ (Launch<LOGM, R>::THREADS, Launch<LOGM, R>::MIN_BLOCKS) istft_kernel (const FftArgs a)
{
    istft_body<LOGM, R, LOGW> (a);
}

// ---------------------------------------------------------------------------------------------
// host side: twiddle tables (fp64 -> fp32), shared by the plan and the emulator tests
// ---------------------------------------------------------------------------------------------
template <int LOGM, int R>
inline void fill_stage_twiddles (float2* tw) // Geo<LOGM,R>::TW_LEN entries, layout described in Geo
{
    using G = Geo<LOGM, R>;
    const long double two_pi = 2.0L * 3.141592653589793238462643383279502884L;
    for (int s = 1; s < G::S; ++s)
    {
        const int r = G::radix (s), Ns = G::ns (s);
        float2* t = tw + G::tw_off (s);
        const long long period = (long long) Ns * r;
        if (r == R)
        {
            const int rows[10] = { 1, 2, 3, 4, 8, 12, 16, 20, 24, 28 };
            for (int i = 0; i < G::FULL_ROWS; ++i)
                for (int k = 0; k < Ns; ++k)
                {
                    const long double ang = -two_pi * (long double) (((long long) k * rows[i]) % period) / (long double) period;
                    t[i * Ns + k] = make_float2 ((float) cosl (ang), (float) sinl (ang));
                }
        }
        else
        {
            for (int q = 1; q < r; ++q)
                for (int k = 0; k < G::T; ++k)
                {
                    const long double ang = -two_pi * (long double) (((long long) k * q) % period) / (long double) period;
                    t[(q - 1) * G::T + k] = make_float2 ((float) cosl (ang), (float) sinl (ang));
                }
        }
    }
}
inline void fill_real_twiddles (float2* rtw, int M) // M/2 entries: exp(-2 pi i k / 2M) / 2 (the split step's 1/2 folded in, exact)
{
    for (int k = 0; k < M / 2; ++k)
    {
        const long double ang = -2.0L * 3.141592653589793238462643383279502884L * (long double) k / (long double) (2LL * M);
        rtw[k] = make_float2 (0.5f * (float) cosl (ang), 0.5f * (float) sinl (ang));
    }
}
} // namespace cfb
