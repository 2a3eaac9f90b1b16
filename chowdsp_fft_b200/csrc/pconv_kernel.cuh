// Fused uniform-partitioned overlap-save convolution step (the "reverb" chain): for every channel
//   X_t   = unordered R2C (window of N samples)            -> written to the frequency-delay line slot t % P
//   Y     = sum_p  X_(t-p) * H_p * scaling                  -> fft_convolve_unordered semantics, P partitions
//   out   = last N/2 samples of unordered C2R (Y)
// in ONE kernel per block step.  It replaces, per channel and block, the reference call sequence
//   fft_transform_unordered (FORWARD) ; P x fft_convolve_unordered ; fft_transform_unordered (BACKWARD)
//   (/root/reference/chowdsp_fft.cpp:358-432, kernels simd/chowdsp_fft_impl_avx.cpp:1848-1979; usage pattern
//    test/test.cpp:214-218) -- 2 + 4 P buffer sweeps through memory -- with a single pass in which the
// accumulator never leaves registers: HBM sees the window once, each delayed spectrum and each IR
// partition once, and N/2 output samples.  Spectra in the delay line and the IR are stored in the
// reference's unordered layout, so they stay interoperable with fft_transform_unordered /
// fft_convolve_unordered.
#pragma once
#include "fft_kernels.cuh"

namespace cfb
{
struct PConvArgs
{
    const float* in;   // channel c's window: in + c * in_stride, N contiguous samples (previous block | new block)
    long long in_stride;
    const float* ir;   // partition p of channel c: ir + c * ir_ch_stride + p * N   (ir_ch_stride = 0: shared IR)
    long long ir_ch_stride;
    float* fdl;        // slot q of channel c: fdl + c * fdl_ch_stride + q * N, q in [0, P)
    long long fdl_ch_stride;
    float* out;        // channel c's N/2 output samples: out + c * out_stride
    long long out_stride;
    int channels;
    int P;             // partitions
    int t;             // block index: slot t % P is written, partitions 0..min(t, P-1) are summed
    float scaling;
    const float2* tw;
    const float2* rtw;
};

FFT_HD float4 ld_stream4 (const float* p) { return ldg_stream (reinterpret_cast<const float4*> (p)); }

// acc += x * h on four lanes (re/im held in separate float4)
FFT_HD void cmac4 (float4& ar, float4& ai, const float4& xr, const float4& xi, const float4& hr, const float4& hi)
{
    ar.x = fmaf (xr.x, hr.x, ar.x); ar.x = fmaf (-xi.x, hi.x, ar.x); ai.x = fmaf (xr.x, hi.x, ai.x); ai.x = fmaf (xi.x, hr.x, ai.x);
    ar.y = fmaf (xr.y, hr.y, ar.y); ar.y = fmaf (-xi.y, hi.y, ar.y); ai.y = fmaf (xr.y, hi.y, ai.y); ai.y = fmaf (xi.y, hr.y, ai.y);
    ar.z = fmaf (xr.z, hr.z, ar.z); ar.z = fmaf (-xi.z, hi.z, ar.z); ai.z = fmaf (xr.z, hi.z, ai.z); ai.z = fmaf (xi.z, hr.z, ai.z);
    ar.w = fmaf (xr.w, hr.w, ar.w); ar.w = fmaf (-xi.w, hi.w, ar.w); ai.w = fmaf (xr.w, hi.w, ai.w); ai.w = fmaf (xi.w, hr.w, ai.w);
}

template <int LOGM>
struct PConvLaunch
{
    using G = Geo<LOGM, 16>;
    // channels per CTA: 256 threads' worth for blocks up to N = 512 (measured on B200, tools/pconv_sweep.py: 2.7x at N = 128, 1.6x at 256, +7 % at 512;
    // from N = 1024 on one channel per CTA is 1..3 % faster and stays)
    static constexpr int PER_CTA = G::T > 16 ? 1 : 256 / G::T;
    static constexpr int THREADS = PER_CTA * G::T;
    static constexpr int SMEM_BYTES = PER_CTA * G::SMEM_F2_UNORD * 8;
};

// Output modes of the fused step (template parameter of pconv_body; PCONV_WRITE is the plain block step above).  The streaming
// convolver (fft_convolver_*) sums segments of different block sizes in a per-channel accumulator ring:
//   PCONV_ADD   out[n] += y[n]                       (a segment's delayed contribution, strictly in the future of the ring)
//   PCONV_EMIT  out[n]  = y[n] + acc[n], acc[n] = 0  (the block being emitted; frees that ring region for later additions)
//   PCONV_EMIT_MIX  out[n] = (1 - g) out[n] + g (y[n] + acc[n]), acc[n] = 0, g = min(mix_start + n mix_step, 1)  (IR crossfade:
//                   the new IR's bank mixed over the output the current bank has just emitted)
// PARTIAL: the accumulator starts from a precomputed partial spectrum S (sum of the older partitions, pconv_slice_kernel) and
// only the newest spectrum X_t (p = 0) is multiplied in here; slot t % P of the delay line is still written.
// FROM_FDL: no forward transform; X_t is read from delay-line slot t % P, which an earlier launch has written, and the slot is
// not written.  The products are those of the fused path, which multiplies the same values from registers, so the result is
// bitwise the same.  A second IR bank (fft_convolver_set_ir) runs this way on the spectra the current bank has just stored.
enum PConvMode
{
    PCONV_WRITE = 0,
    PCONV_ADD = 1,
    PCONV_EMIT = 2,
    PCONV_EMIT_MIX = 3
};

struct PConvAcc
{
    float* acc;         // PCONV_EMIT / PCONV_EMIT_MIX: channel c's ring region at acc + c * acc_stride (N/2 samples)
    long long acc_stride;
    const float* S;     // PARTIAL: channel c's partial spectrum at S + c * s_stride (N floats, unordered, unscaled)
    long long s_stride;
    float mix_start, mix_step; // PCONV_EMIT_MIX: weight of the new result at output sample 0 and its step per sample
};

template <int LOGM, int LOGW, int MODE = PCONV_WRITE, bool PARTIAL = false, bool FROM_FDL = false>
FFT_HD void pconv_body (const PConvArgs& a, const PConvAcc& x = PConvAcc {})
{
    constexpr int R = 16;
    using G = Geo<LOGM, R>;
    constexpr int M = G::M, T = G::T, N = 2 * M, W = 1 << LOGW;
    constexpr int PAIRS = R / 4; // (4 re | 4 im) lane groups per thread: N / 8 per spectrum = 4 T
    // small blocks: a CTA of 256 threads takes 256 / T channels (one channel per CTA left 4 .. 128-thread CTAs for N <= 4096);
    // channels past the end redo the last one and skip every global store (the barriers inside fft_core are CTA-wide)
    constexpr int PER_CTA = PConvLaunch<LOGM>::PER_CTA;
    FFT_DYN_SMEM (float2, smem_all);
    const int lt = PER_CTA == 1 ? 0 : (int) threadIdx.x / T, j = (int) threadIdx.x - lt * T;
    float2* smem = smem_all + lt * G::SMEM_F2_UNORD;
    float* sf = reinterpret_cast<float*> (smem);
    const long long c0 = (long long) blockIdx.x * PER_CTA + lt;
    const bool active = PER_CTA == 1 || c0 < a.channels;
    const int c = active ? (int) c0 : a.channels - 1;

    // 1. forward transform of the window; the unordered spectrum stays in shared memory (staging image)
    if constexpr (! FROM_FDL)
        fft_core<LOGM, R, R2C, LOGW, false, true, false> (a.in + (long long) c * a.in_stride, nullptr, true, j, smem, a.tw, a.rtw);

    // 2. this thread's slice of the spectrum: PAIRS x (4 re lanes, 4 im lanes); float offset of the re quad
    int off[PAIRS];
    float4 xr[PAIRS], xi[PAIRS], ar[PAIRS], ai[PAIRS];
    float* slot = a.fdl + (long long) c * a.fdl_ch_stride + (long long) (a.t % a.P) * N;
#pragma unroll
    for (int i = 0; i < PAIRS; ++i)
    {
        const int pr = j + i * T;
        off[i] = (pr / (W / 4)) * 2 * W + (pr % (W / 4)) * 4;
        if constexpr (FROM_FDL)
        {
            xr[i] = ld_stream4 (slot + off[i]);
            xi[i] = ld_stream4 (slot + off[i] + W);
        }
        else
        {
            xr[i] = lds4 (sf + upad (off[i], LOGW));
            xi[i] = lds4 (sf + upad (off[i] + W, LOGW));
            if (active)
            {
                *reinterpret_cast<float4*> (slot + off[i]) = xr[i];     // delay-line write (linear across the channel's threads)
                *reinterpret_cast<float4*> (slot + off[i] + W) = xi[i];
            }
        }
        if constexpr (PARTIAL)
        {
            const float* sc = x.S + (long long) c * x.s_stride;
            ar[i] = ld_stream4 (sc + off[i]);
            ai[i] = ld_stream4 (sc + off[i] + W);
        }
        else
        {
            ar[i] = make_float4 (0.f, 0.f, 0.f, 0.f);
            ai[i] = make_float4 (0.f, 0.f, 0.f, 0.f);
        }
    }

    // 3. frequency-domain multiply-accumulate over the partitions; DC / Nyquist (float slots 0 and W of a
    //    real spectrum, lane 0 of this CTA's first pair) are two independent REAL products
    float dc = PARTIAL ? ar[0].x : 0.f, ny = PARTIAL ? ai[0].x : 0.f;
    const float* irc = a.ir + (long long) c * a.ir_ch_stride;
    const float* fdlc = a.fdl + (long long) c * a.fdl_ch_stride;
    const int np = PARTIAL ? 1 : (a.t + 1 < a.P ? a.t + 1 : a.P);
    for (int p = 0; p < np; ++p)
    {
        const float* h = irc + (long long) p * N;
        int q = (a.t - p) % a.P;
        const float* xs = fdlc + (long long) q * N;
        float4 hr[PAIRS], hi[PAIRS];
#pragma unroll
        for (int i = 0; i < PAIRS; ++i)
        {
            hr[i] = ld_stream4 (h + off[i]);
            hi[i] = ld_stream4 (h + off[i] + W);
        }
        if (p > 0) // p == 0 is the spectrum just computed, still in registers
        {
#pragma unroll
            for (int i = 0; i < PAIRS; ++i)
            {
                xr[i] = ld_stream4 (xs + off[i]);
                xi[i] = ld_stream4 (xs + off[i] + W);
            }
        }
        dc = fmaf (xr[0].x, hr[0].x, dc);
        ny = fmaf (xi[0].x, hi[0].x, ny);
#pragma unroll
        for (int i = 0; i < PAIRS; ++i)
            cmac4 (ar[i], ai[i], xr[i], xi[i], hr[i], hi[i]);
    }
    if (j == 0)
    {
        ar[0].x = dc;
        ai[0].x = ny;
    }

    // 4. scaled accumulator becomes the staging image of the inverse transform
    __syncthreads(); // every thread has taken its slice of X_t out of the staging image
    const float sc = a.scaling;
#pragma unroll
    for (int i = 0; i < PAIRS; ++i)
    {
        sts4 (sf + upad (off[i], LOGW), make_float4 (ar[i].x * sc, ar[i].y * sc, ar[i].z * sc, ar[i].w * sc));
        sts4 (sf + upad (off[i] + W, LOGW), make_float4 (ai[i].x * sc, ai[i].y * sc, ai[i].z * sc, ai[i].w * sc));
    }
    __syncthreads();

    // 5. inverse transform; only the last N/2 samples are valid in overlap-save and only they are stored
    float* outc = a.out + (long long) c * a.out_stride - M; // sample n >= M lands at out[n - M]
    if constexpr (MODE == PCONV_WRITE)
        fft_core<LOGM, R, C2R, LOGW, true, false, true> (nullptr, outc, active, j, smem, a.tw, a.rtw);
    else
    {
        // the same inverse transform with the result handed back in registers (element j + m T in v[m]); the store adds
        float2 v[R];
        fft_core<LOGM, R, C2R, LOGW, true, false, true, 0, NoHook, true> (nullptr, nullptr, active, j, smem, a.tw, a.rtw, nullptr, nullptr, NoHook(), v);
        if (active)
        {
            float2* o2 = reinterpret_cast<float2*> (outc) + j;
            float2* acc2 = MODE != PCONV_ADD ? reinterpret_cast<float2*> (x.acc + (long long) c * x.acc_stride - M) + j : nullptr;
#pragma unroll
            for (int m = R / 2; m < R; ++m)
            {
                if constexpr (MODE == PCONV_ADD)
                    o2[m * T] = f2_add (o2[m * T], v[m]);
                else if constexpr (MODE == PCONV_EMIT)
                {
                    o2[m * T] = f2_add (v[m], acc2[m * T]);
                    acc2[m * T] = make_float2 (0.f, 0.f);
                }
                else
                {
                    const float2 r = f2_add (v[m], acc2[m * T]), o = o2[m * T];
                    const float n = (float) (2 * (j + m * T) - M); // output sample of r.x
                    const float g0 = fminf (fmaf (n, x.mix_step, x.mix_start), 1.f), g1 = fminf (fmaf (n + 1.f, x.mix_step, x.mix_start), 1.f);
                    o2[m * T] = make_float2 (fmaf (g0, r.x, (1.f - g0) * o.x), fmaf (g1, r.y, (1.f - g1) * o.y));
                    acc2[m * T] = make_float2 (0.f, 0.f);
                }
            }
        }
    }
}

template <int LOGM, int LOGW>
__global__ void __launch_bounds__ (PConvLaunch<LOGM>::THREADS, (PConvLaunch<LOGM>::THREADS <= 256 ? 2 : 1)) pconv_kernel (const PConvArgs a)
{
    pconv_body<LOGM, LOGW> (a);
}

// the accumulating modes (streaming convolver): one instance per (MODE, PARTIAL, FROM_FDL) in use
template <int LOGM, int LOGW, int MODE, bool PARTIAL, bool FROM_FDL = false>
__global__ void __launch_bounds__ (PConvLaunch<LOGM>::THREADS, (PConvLaunch<LOGM>::THREADS <= 256 ? 2 : 1)) pconv_acc_kernel (const PConvArgs a, const PConvAcc x)
{
    pconv_body<LOGM, LOGW, MODE, PARTIAL, FROM_FDL> (a, x);
}

// ---------------------------------------------------------------------------------------------
// Sliced tail multiply-accumulate of the streaming convolver (pconv_slice_kernel, elementwise_kernels.cuh): the part of a P-partition segment's spectral sum that does not
// depend on the newest block,  S = sum_{p=1}^{P-1} X_(q-p) * H_p  (X_g in delay-line slot g % P, unscaled), for one slice of
// the spectrum -- pairs [pair0, pair0 + pairs), a pair being 4 re lanes at float offset off and their 4 im lanes at off + W.
// Spread over the small steps between two firings of the segment, every bin of S is written once per period and the firing
// itself (pconv_acc_kernel<.., PARTIAL>) only multiplies X_q * H_0.  Same products and real DC / Nyquist lanes as pconv_body.
struct PConvSliceArgs
{
    const float* ir;   // partition p of channel c: ir + c * ir_ch_stride + p * N
    long long ir_ch_stride;
    const float* fdl;  // slot g of channel c: fdl + c * fdl_ch_stride + g * N
    long long fdl_ch_stride;
    float* S;          // channel c's partial spectrum: S + c * s_stride
    long long s_stride;
    int channels;
    int P;
    int N;
    int logW;
    int q;             // the firing S is for
    int pair0, pairs;
};

// Non-uniform partition schedule of the streaming convolver (host code; the emulator driver exposes it to the tests).  For
// block B, IR length L and largest block Bmax (>= B):  segment 0 has block B and 2 partitions (taps [0, 2B)); segment k >= 1
// has block Bk = 2^k B and one partition (taps [Bk, 2 Bk), output delay Bk) until Bk = Bmax, which takes the rest of the IR
// in ceil((L - Bmax) / Bmax) partitions; the schedule stops as soon as the IR is covered.  L <= 2B or Bmax == B: one uniform
// segment of ceil(L / B) partitions.  Writes up to max_segments (block, partitions, first tap) entries; returns the count.
inline int conv_schedule (int B, long long L, int Bmax, int* block, long long* parts, long long* start, int max_segments)
{
    int n = 0;
    auto put = [&] (int bk, long long p, long long s0)
    {
        if (n < max_segments)
        {
            block[n] = bk;
            parts[n] = p;
            start[n] = s0;
        }
        ++n;
    };
    if (L <= 2LL * B || Bmax <= B)
    {
        put (B, (L + B - 1) / B, 0);
        return n;
    }
    put (B, 2, 0);
    for (long long bk = 2LL * B; bk < L; bk *= 2)
    {
        if (bk >= Bmax)
        {
            put ((int) bk, (L - bk + bk - 1) / bk, bk);
            break;
        }
        put ((int) bk, 1, bk);
    }
    return n;
}

// The convolver's input history (conv_input_kernel, elementwise_kernels.cuh): each channel's new block of B samples is written at pos and again at pos + mirror of a
// mirrored ring (2 x mirror floats per channel), so that every window -- the last 2 B_k samples -- is one contiguous span.
struct ConvInputArgs
{
    const float* in;   // channel c's block: in + c * in_stride, B samples (8-byte aligned, even stride)
    long long in_stride;
    float* hist;       // channel c's ring: hist + c * hist_stride
    long long hist_stride;
    int channels;
    int half_block;    // B / 2 float2 per channel
    long long pos, mirror;
};

// IR preparation (conv_ir_gather_kernel, elementwise_kernels.cuh; at context creation, not on the streaming path): partition p of channel c of a segment with block Bk,
// starting at tap `start`, as the zero-padded window [Bk taps | Bk zeros] at dst + (c * P + p) * 2 Bk; taps past `length`
// are zeros.  The forward transform of these windows is done by the ordinary batched transform.
struct ConvIrArgs
{
    const float* ir;
    long long ir_stride;
    float* dst;
    long long length, start;
    int channels, P, Bk;
};

} // namespace cfb
